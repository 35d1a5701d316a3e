"""bench.py --dump-outputs: the arrays the last timed step returned, written so that two builds can be compared output
for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path, monkeypatch):
    import bench
    B = 1000
    arrays = {'obs': np.arange(4 * B, dtype=np.float32).reshape(B, 4), 'reward': np.arange(B, dtype=np.float64) / 7}
    bench.dump_outputs(arrays, str(tmp_path / 'whole'))
    assert sorted(os.listdir(tmp_path / 'whole')) == ['obs.npy', 'reward.npy']
    assert np.array_equal(np.load(tmp_path / 'whole' / 'obs.npy'), arrays['obs'])
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 4096 + 12000)       # room for 375 of the 1000 rows and their indices
    for d in ('a', 'b'):
        bench.dump_outputs(arrays, str(tmp_path / d))
    got = [{n: np.load(tmp_path / d / (n + '.npy')) for n in ('obs', 'reward', 'env_index')} for d in ('a', 'b')]
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= bench.DUMP_LIMIT
    idx = got[0]['env_index']
    assert idx.dtype == np.float64 and len(idx) == 375 and np.all(np.diff(idx) > 0)
    rows = idx.astype(np.int64)
    assert np.array_equal(got[0]['obs'], arrays['obs'][rows]) and np.array_equal(got[0]['reward'], arrays['reward'][rows])
    for n in got[0]:
        assert np.array_equal(got[0][n], got[1][n])


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """The dump is the result of the last of --steps timed steps: an AOVecEnv driven independently through the same
    seeds, episode phase, warm-up and 7 steps ends in the same outputs, and one step more does not."""
    import torch
    import bench
    from adaptive_optics_gym_b200 import AOVecEnv
    B, warmup, steps = 64, 3, 7
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--envs', str(B), '--steps',
                          str(steps), '--warmup', str(warmup), '--no-cpu-baseline', '--no-mft-arm', '--no-workloads',
                          '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    names = ('obs', 'obs_f64', 'reward', 'power', 'done')
    assert sorted(os.listdir(tmp_path)) == sorted(n + '.npy' for n in names)
    dump = {n: np.load(tmp_path / (n + '.npy')) for n in names}
    assert dump['obs'].dtype == dump['done'].dtype == np.float32 and dump['obs_f64'].dtype == np.float64

    # bench.Runner: env seed 1234, a pool of 8 action batches from CPU generator seed 7, the episode clock phased so
    # that an episode end falls inside the timed window, a reset at every episode boundary
    w = bench.WORKLOADS['quasi_static_64act']
    T = w['timesteps_per_episode']
    env = AOVecEnv(B, **w, device=0, seed=1234, precision='fused')
    g = torch.Generator(device='cpu').manual_seed(7)
    acts = [torch.empty((B, 64), dtype=torch.float32).uniform_(-1, 1, generator=g).cuda() for _ in range(8)]
    pre = (T - (warmup + max(steps // 2, 1))) % T
    env.reset()
    env._h.set_counters(timestep_render=pre)
    t, resets = (pre if pre else T), 0

    def step(i):
        nonlocal t, resets
        if t % T == 0:
            env.reset()
            resets += 1
        obs, rew, done, _, info = env.step(acts[i % len(acts)])
        t += 1
        return {'obs': obs.float(), 'obs_f64': env.obs_f64, 'reward': rew, 'power': info['power'], 'done': done.float()}

    for i in range(warmup + steps):
        got = {n: v.cpu().numpy() for n, v in step(i).items()}
    assert resets == 1                                   # the window crossed an episode end
    for n in names:
        assert np.array_equal(got[n], dump[n]), n
    after = step(warmup + steps)
    assert not np.array_equal(after['obs_f64'].cpu().numpy(), dump['obs_f64'])
    env.close()
