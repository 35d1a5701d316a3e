"""The reference's OWN callers, unmodified, against this repo's ``gym_AO`` on a B200.

``main.py:280-292`` (the ``gym.make('AO-v0', ...)`` call with its literal kwargs), ``main.py:25-85`` (``train``),
``algorithm.py:22-143`` (``ALGORITHM.__init__``), ``algorithm.py:216-296`` (``rollout``: ``env.reset`` /
``env.render`` / ``actor.get_action`` or ``env.SH_step`` / ``env.step``) and ``eval_policy.py:8-43`` run exactly as
the reference wrote them; only ``ALGORITHM.learn`` is replaced by "one rollout" so the test ends in seconds, and
``gymnasium`` / ``matplotlib`` (absent from this image) are stood in for by ``_gym_compat`` and a no-op stub.

The caller files are the reference project's own sources, which this repository does not carry: they are looked up
in ``$AOG_REFERENCE_DIR`` or ``baseline/_ref/callers`` (``tools/stage_reference_callers.py``; git-ignored), the test
skips without them, and they must match the committed SHA-256 manifest -- no reference file is edited.  Our
``gym_AO`` sits AHEAD of the reference's on ``sys.path``.
"""
import argparse
import hashlib
import importlib
import os
import sys
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLERS = ['main.py', 'algorithm.py', 'network.py', 'replay_buffer.py', 'eval_policy.py', 'arguments.py']


def _find_callers():
    for d in (os.environ.get('AOG_REFERENCE_DIR'), os.path.join(ROOT, 'baseline', '_ref', 'callers')):
        if d and all(os.path.exists(os.path.join(d, f)) for f in CALLERS):
            return d
    return None


class _Anything(types.ModuleType):
    """matplotlib stand-in: every attribute is a callable that returns another stand-in."""

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        return _Anything(name)

    def __call__(self, *a, **k):
        return _Anything('result')

    def __iter__(self):
        return iter(())


@pytest.fixture()
def reference(monkeypatch):
    d = _find_callers()
    if d is None:
        pytest.skip('reference callers not staged (python tools/stage_reference_callers.py)')
    want = dict(line.split()[::-1] for line in open(os.path.join(ROOT, 'tests', 'golden', 'reference_callers.sha256')))
    for f in CALLERS:
        assert hashlib.sha256(open(os.path.join(d, f), 'rb').read()).hexdigest() == want[f], f'{f} is not the reference file'
    from adaptive_optics_gym_b200 import _gym_compat as G
    if not G.HAVE_GYMNASIUM:        # `import gymnasium as gym`, `gym.spaces.Box`, `gym.make`, registration.register
        gymn = types.ModuleType('gymnasium')
        gymn.spaces, gymn.make, gymn.Env = G.spaces, G.make, G.Env
        reg = types.ModuleType('gymnasium.envs.registration')
        reg.register = G.register
        envs = types.ModuleType('gymnasium.envs')
        envs.registration = reg
        gymn.envs = envs
        for name, mod in (('gymnasium', gymn), ('gymnasium.envs', envs), ('gymnasium.envs.registration', reg)):
            monkeypatch.setitem(sys.modules, name, mod)
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        mpl = _Anything('matplotlib')
        monkeypatch.setitem(sys.modules, 'matplotlib', mpl)
        monkeypatch.setitem(sys.modules, 'matplotlib.pyplot', _Anything('matplotlib.pyplot'))
    # our gym_AO first, the reference directory LAST (it carries its own gym_AO package)
    monkeypatch.setattr(sys, 'path', [ROOT] + [p for p in sys.path if p not in (ROOT, d)] + [d])
    for name in ('main', 'algorithm', 'network', 'replay_buffer', 'eval_policy', 'arguments'):
        monkeypatch.delitem(sys.modules, name, raising=False)
    import gym_AO
    assert os.path.dirname(os.path.abspath(gym_AO.__file__)) == os.path.join(ROOT, 'gym_AO')
    main = importlib.import_module('main')
    assert os.path.samefile(os.path.dirname(main.__file__), d)
    return main


def _args(algo):
    return argparse.Namespace(mode='train', environment_name='AO-v0', algorithm_name=algo, actor_model='',
                              criticQ1_model='', criticQ2_model='', criticV_model='')


@pytest.mark.parametrize('algo,episodes', [('PPO', 2), ('DDPG', 2), ('SAC', 1), ('SHACK', 1)])
@pytest.mark.parametrize('precision', ['f64', 'fused'])
def test_reference_main_train_rollout_runs_unchanged(reference, monkeypatch, algo, episodes, precision):
    main = reference
    from adaptive_optics_gym_b200 import AOEnv
    monkeypatch.setenv('AOG_PRECISION', precision)       # main.py passes only the reference's kwargs
    got = {}

    def one_rollout(self, total_timesteps):              # stands in for ALGORITHM.learn (algorithm.py:146-210)
        self.num_episodes = 0
        self.epoch_no = 0
        got['model'] = self
        got['batches'] = self.rollout()                  # algorithm.py:216-296, unchanged

    monkeypatch.setattr(main.ALGORITHM, 'learn', one_rollout)
    main.main(_args(algo))                               # main.py:137-300: literal dicts, gym.make, train()
    model = got['model']
    env = model.env
    assert isinstance(env, AOEnv) and env.precision == precision
    assert env.SH_operation == (algo == 'SHACK') and env.max_steps == 30 and env.num_modes == 64
    T = episodes * 30
    obs, act, logp, rew, nobs, done, lens = got['batches']
    import torch
    for t, shape in ((obs, (T, 4)), (act, (T, 64)), (logp, (T,)), (rew, (T,)), (nobs, (T, 4)), (done, (T,))):
        assert tuple(t.shape) == shape and t.dtype == torch.float32
    assert lens.shape == (T,) and list(lens[:episodes]) == [30.0] * episodes
    assert torch.isfinite(obs).all() and torch.isfinite(rew).all() and torch.isfinite(act).all()
    assert done.sum().item() == episodes and all(done[30 * (k + 1) - 1] == 1 for k in range(episodes))
    assert torch.equal(obs[1:30], nobs[:29])             # next_obs of step t is obs of step t + 1 within an episode
    assert (rew <= 0).all() and (rew >= -100).all()      # strehl_ratio reward = -(100 - Strehl %)
    assert env.episode_no == episodes and env.timestep == T
    if algo == 'SHACK':
        assert (logp == 1).all()                         # AO_env.py:290 returns torch.tensor([1]) as the "log prob"
        assert rew[-1] > rew[0]                          # the integrator closes the loop on a static atmosphere
    if algo != 'SHACK':
        # eval_policy.py:8-43, unchanged: one evaluation episode with the actor main.py built
        ev = importlib.import_module('eval_policy')
        ep_len, ep_ret = next(ev.rollout(model.actor, env, True))
        assert ep_len == 30 and np.isfinite(ep_ret) and isinstance(env.last_render['focal_power'], np.ndarray)
    env.close()
