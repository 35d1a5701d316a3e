"""GPU: a Fried parameter per env (``AOVecEnv(atm_fried=[...])``, ``reset(options={'atm_fried': ...})``,
``aog_set_turbulence``).  Each env's arithmetic reads only its own screen and its own sqrt(Cn^2), so a mixed batch must
reproduce, bit for bit, handles built with one scalar r0 each."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R0_MIX = [0.05, 0.08, 0.10, 0.20] * 2


def _kw(atm_type, **extra):
    kw = dict(atm_type=atm_type, atm_vel=20 if atm_type == 'dynamic' else 0, act_dim=64, obs_dim=2,
              rew_type='strehl_ratio', timesteps_per_episode=3)
    kw.update(extra)
    return kw


def _actions(B, seed):
    import torch
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.rand((B, 64), generator=g) * 2 - 1).cuda()


def _outputs(env):
    """(float16 obs bits, reward, power) of the last step / reset on the host"""
    import torch
    torch.cuda.synchronize()
    return (env.obs.cpu().numpy().view(np.uint16).copy(), env.reward.cpu().numpy().copy(),
            env.power.cpu().numpy().copy())


def _screen(seed, r0, n=240):
    from oracle.ao_oracle import hcipy_make_pupil_grid, hcipy_Cn_squared_from_fried_parameter, von_karman_screen
    g = hcipy_make_pupil_grid(n, 0.5)
    return von_karman_screen(g, hcipy_Cn_squared_from_fried_parameter(r0, 2.2e-6), 10.0, np.random.default_rng(seed))


def _close_obs(got, want, what):
    """detector powers at the tolerance of tests/test_parity_gpu.py::_close_obs (1e-5 relative + amplitude floor)"""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    peak = want.max(axis=-1, keepdims=True)
    tol = 1e-5 * want + 2e-8 * np.sqrt(want * peak)
    assert np.all(np.abs(got - want) <= tol), what


@pytest.mark.parametrize('atm_type', ['quasi_static', 'semi_dynamic', 'dynamic'])
@pytest.mark.parametrize('precision', ['f64', 'tensor', 'fused'])
def test_mixed_batch_equals_scalar_handles(precision, atm_type):
    from adaptive_optics_gym_b200 import AOVecEnv
    B = len(R0_MIX)
    kw = _kw(atm_type, seed=5, precision=precision)
    mixed = AOVecEnv(B, atm_fried=R0_MIX, **kw)
    assert isinstance(mixed.fried_parameter, np.ndarray) and mixed.fried_parameter.tolist() == R0_MIX
    scalar = {r: AOVecEnv(B, atm_fried=r, **kw) for r in sorted(set(R0_MIX))}
    assert isinstance(scalar[0.05].fried_parameter, float)
    everyone = [mixed] + list(scalar.values())

    def check(what, get):
        got = get(mixed)
        want = {r: get(e) for r, e in scalar.items()}
        for i, r in enumerate(R0_MIX):
            for g, w in zip(got, want[r]):
                assert np.array_equal(g[i], w[i]), f'{what}: env {i} (r0 = {r}) differs from the scalar handle'

    check('screens after construction', lambda e: (e._h.get_screens(),))
    for ep in range(2):
        for e in everyone:
            e.reset()
        check(f'reset {ep}', lambda e: _outputs(e)[:1] + (e._h.get_screens(),))
        for t in range(3):
            a = _actions(B, 10 * ep + t)
            for e in everyone:
                e.step(a)
            check(f'episode {ep} step {t}', lambda e: _outputs(e) + (e._h.get_screens(),))
    if atm_type == 'dynamic':
        assert mixed._h.counters().extrusions >= 50           # 6 steps at 9.6 px each, device Philox noise
    for e in everyone:
        e.close()


@pytest.mark.parametrize('precision', ['f64', 'tensor', 'fused'])
def test_dynamic_injected_noise_against_oracles(precision):
    """dynamic, v = 20 m/s, r0 = (0.06, 0.10, 0.20) in one handle against three oracles: same AR tables, initial
    screens and normals; env i follows the AR process of its own r0."""
    import torch
    from adaptive_optics_gym_b200 import AOVecEnv
    from oracle.ao_oracle import OracleAOEnv
    r0 = (0.06, 0.10, 0.20)
    kw = dict(atm_type='dynamic', atm_vel=20, act_dim=64, obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=3)
    scr = [_screen(30 + i, r) for i, r in enumerate(r0)]
    refs = [OracleAOEnv(**kw, atm_fried=r, initial_screen=s, seed=11) for r, s in zip(r0, scr)]
    lay = refs[0].layer
    tabs = dict(ar_stencil=np.flatnonzero(lay.stencil_left).astype(np.int32), ar_A=lay.A_horizontal,
                ar_B=lay.B_horizontal)
    for ref in refs[1:]:        # the AR operator does not depend on r0 (it is built at Cn^2 = 1)
        assert np.array_equal(ref.layer.stencil_left, lay.stencil_left)
        assert np.array_equal(ref.layer.A_horizontal, lay.A_horizontal)
        assert np.array_equal(ref.layer.B_horizontal, lay.B_horizontal)
    env = AOVecEnv(3, **kw, atm_fried=list(r0), initial_screens=np.stack(scr), tables=tabs, precision=precision)
    rtol = 1e-7 if precision == 'f64' else 1e-5
    rng = np.random.default_rng(8)
    for ep in range(2):
        env.reset()
        for ref in refs:
            ref.reset()
        for t in range(3):
            n_ext = refs[0].num_extrusions_for_next_step()
            noise = rng.standard_normal((3, n_ext, 240))
            a = rng.uniform(-1, 1, (3, 64)).astype(np.float32)
            env.step(torch.from_numpy(a).cuda(), extrusion_noise=noise)
            got = _outputs(env)
            s_gpu = env._h.get_screens()
            obs = env.obs_f64.cpu().numpy()
            for i, ref in enumerate(refs):
                _, rr, _, _, rinfo = ref.step(a[i], extrusion_noise=noise[i])
                want = ref.layer.achromatic_screen
                np.testing.assert_allclose(s_gpu[i], want, rtol=0, atol=1e-9 * np.abs(want).max())
                if precision == 'f64':
                    np.testing.assert_allclose(obs[i], ref.last_obs_f64, rtol=rtol)
                else:
                    _close_obs(obs[i], ref.last_obs_f64, f'obs env {i}')
                np.testing.assert_allclose(got[1][i], rr, rtol=rtol)
                np.testing.assert_allclose(got[2][i], rinfo['power'], rtol=rtol)
    env.close()


def test_generated_screens_statistics_per_env():
    """semi_dynamic synthesis with two r0 in one batch: each half's structure function follows the von Karman value
    of its own r0 (as test_generated_screens_statistics_and_semi_dynamic does for one r0); and the largest phase stays
    inside the budget behind tables.FRIED_MIN (100 rad at r0 = 0.20 m, scaled by r0^(-5/6))."""
    from adaptive_optics_gym_b200 import AOVecEnv
    from oracle.ao_oracle import (hcipy_Cn_squared_from_fried_parameter, hcipy_fried_parameter_from_Cn_squared,
                                  hcipy_phase_covariance_von_karman)
    B = 192
    r0 = np.array([0.08] * (B // 2) + [0.20] * (B // 2))
    env = AOVecEnv(B, atm_type='semi_dynamic', atm_fried=r0, seed=3)
    s0 = env._h.get_screens().reshape(B, 240, 240)
    env.reset()
    s1 = env._h.get_screens().reshape(B, 240, 240)
    d = 0.5 / 240
    for half, r in ((slice(0, B // 2), 0.08), (slice(B // 2, B), 0.20)):
        cn2 = hcipy_Cn_squared_from_fried_parameter(r, 2.2e-6)
        cov = hcipy_phase_covariance_von_karman(hcipy_fried_parameter_from_Cn_squared(cn2, 1.0), 10.0)
        for lag in (4, 16, 64):
            th = 2 * (cov(np.array(0.0)) - cov(np.array(lag * d)))
            for s in (s0[half], s1[half]):
                dx = np.mean((s[:, :, lag:] - s[:, :, :-lag]) ** 2)
                dy = np.mean((s[:, lag:, :] - s[:, :-lag, :]) ** 2)
                assert 0.85 < dx / th < 1.15 and 0.85 < dy / th < 1.15, (r, lag, dx / th, dy / th)
    largest = np.maximum(np.abs(s0).max(axis=(1, 2)), np.abs(s1).max(axis=(1, 2)))
    at_020 = largest * (r0 / 0.20) ** (5 / 6) / env.wavelength_wfs
    assert at_020.max() < 100.0, at_020.max()
    env.close()


@pytest.mark.parametrize('atm_type', ['quasi_static', 'dynamic'])
@pytest.mark.parametrize('precision', ['f64', 'tensor', 'fused'])
def test_reset_option_rescales_kept_screens(precision, atm_type):
    """quasi_static / dynamic: reset(options={'atm_fried': r0_new}) scales each env's screen by (r0_old / r0_new)^(5/6);
    the next steps equal a fresh handle given the rescaled screens (and, on the tensor / fused paths, the rescale pass's
    phase tiles equal the ones a fresh upload computes)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    B = 6
    r0_old = np.array([0.05, 0.08, 0.10, 0.20, 0.15, 0.12])
    r0_new = np.array([0.10, 0.05, 0.20, 0.08, 0.15, 0.30])
    kw = _kw(atm_type, seed=7, precision=precision)
    env = AOVecEnv(B, atm_fried=r0_old, **kw)
    env.reset()
    if atm_type == 'dynamic':
        for t in range(2):                       # move the ring origin away from 0
            env.step(_actions(B, t))
        assert env._h.counters().column_origin != 0
    before = env._h.get_screens()
    env.reset(options={'atm_fried': r0_new})
    assert env.fried_parameter.tolist() == r0_new.tolist()
    after = env._h.get_screens()
    want = before * ((r0_old / r0_new) ** (5 / 6))[:, None]
    assert np.all(np.abs(after - want) <= 1e-14 * np.abs(want))
    reset_out = _outputs(env)

    st = env.get_state()
    if atm_type == 'quasi_static':
        fresh = AOVecEnv(B, atm_fried=r0_new, **kw, initial_screens=after)
        fresh.reset()
        assert np.array_equal(_outputs(fresh)[0], reset_out[0]), 'reset obs'
    else:
        fresh = AOVecEnv(B, atm_fried=r0_new, **kw)
        fresh.set_state(st)                      # same time, draw counters and screens; ring origin 0
    for t in range(3):
        a = _actions(B, 20 + t)
        env.step(a)
        fresh.step(a)
        got, ref = _outputs(env), _outputs(fresh)
        if atm_type == 'quasi_static':
            for g, w in zip(got, ref):
                assert np.array_equal(g, w), f'step {t}'
        else:
            rtol = 1e-7 if precision == 'f64' else 1e-5
            s, s_ref = env._h.get_screens(), fresh._h.get_screens()
            np.testing.assert_allclose(s, s_ref, rtol=0, atol=1e-12 * np.abs(s_ref).max())
            _close_obs(env.obs_f64.cpu().numpy(), fresh.obs_f64.cpu().numpy(), f'obs step {t}')
            np.testing.assert_allclose(got[1], ref[1], rtol=rtol)
            np.testing.assert_allclose(got[2], ref[2], rtol=rtol)
    env.close(), fresh.close()


def test_reset_option_rescale_reaches_the_shack_hartmann_tensor_step():
    from adaptive_optics_gym_b200 import AOVecEnv
    B = 9
    r0_old = np.linspace(0.06, 0.20, B)
    r0_new = r0_old[::-1].copy()
    kw = _kw('quasi_static', seed=4, precision='fused', SH_operation=True)
    env = AOVecEnv(B, atm_fried=r0_old, **kw)
    env.reset(options={'atm_fried': r0_new})
    fresh = AOVecEnv(B, atm_fried=r0_new, **kw, initial_screens=env._h.get_screens())
    fresh.reset()
    for t in range(2):
        a, _ = env.SH_step(noise='none')
        b, _ = fresh.SH_step(noise='none')
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()), f'SH action {t}'
        env.step(a)
        fresh.step(b)
        for g, w in zip(_outputs(env), _outputs(fresh)):
            assert np.array_equal(g, w)
    env.close(), fresh.close()


@pytest.mark.parametrize('precision', ['f64', 'fused'])
def test_reset_option_semi_dynamic_draws_at_the_new_strength(precision):
    from adaptive_optics_gym_b200 import AOVecEnv
    r0_old, r0_new = [0.20, 0.05, 0.10, 0.08], [0.05, 0.20, 0.08, 0.10]
    kw = _kw('semi_dynamic', seed=9, precision=precision)
    env = AOVecEnv(4, atm_fried=r0_old, **kw)
    env.reset(options={'atm_fried': r0_new})
    got = env._h.get_screens()
    for i, r in enumerate(r0_new):
        ref = AOVecEnv(4, atm_fried=r, **kw)
        ref.reset()                                   # the same draw (the second) of the same Philox stream
        assert np.array_equal(got[i], ref._h.get_screens()[i]), f'env {i}'
        ref.close()
    env.close()


def test_reset_without_options_changes_nothing():
    from adaptive_optics_gym_b200 import AOVecEnv
    for atm_type in ('quasi_static', 'dynamic'):
        env = AOVecEnv(4, atm_fried=[0.05, 0.08, 0.10, 0.20], **_kw(atm_type, seed=2, precision='fused'))
        s = env._h.get_screens()
        for opts in (None, {}, {'unrelated': 1}):
            env.reset(options=opts)
            assert np.array_equal(env._h.get_screens(), s)
            assert env.fried_parameter.tolist() == [0.05, 0.08, 0.10, 0.20]
        env.close()


def test_sharding_invariance_with_mixed_r0():
    """two halves with env_id_base and their slices of r0 == the whole batch (synthesis at construction and reset,
    device-Philox extrusions)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    from adaptive_optics_gym_b200.sharding import shard_range
    B = 6
    r0 = np.array([0.05, 0.20, 0.08, 0.10, 0.15, 0.06])
    kw = _kw('dynamic', seed=12, precision='fused')
    whole = AOVecEnv(B, atm_fried=r0, **kw)
    parts = []
    for rank in range(2):
        first, count = shard_range(B, rank, 2)
        parts.append((first, count, AOVecEnv(count, atm_fried=r0[first:first + count], env_id_base=first, **kw)))
    for t in range(4):
        a = _actions(B, t)
        if t == 0:
            whole.reset()
        else:
            whole.step(a)
        n = 1 if t == 0 else 3                       # a reset writes obs only
        got = _outputs(whole)[:n] + (whole._h.get_screens(),)
        for first, count, p in parts:
            if t == 0:
                p.reset()
            else:
                p.step(a[first:first + count])
            for g, w in zip(got, _outputs(p)[:n] + (p._h.get_screens(),)):
                assert np.array_equal(g[first:first + count], w), f'step {t}, shard at {first}'
    whole.close()
    for *_, p in parts:
        p.close()


def test_state_round_trip_carries_the_fried_parameters():
    from adaptive_optics_gym_b200 import AOVecEnv
    B = 5
    r0_a = np.array([0.05, 0.20, 0.08, 0.10, 0.15])
    r0_b = np.array([0.12, 0.12, 0.30, 0.07, 0.09])
    kw = _kw('dynamic', seed=6, precision='fused')
    a = AOVecEnv(B, atm_fried=r0_a, **kw)
    a.reset()
    for t in range(2):
        a.step(_actions(B, t))
    st = a.get_state()
    assert st['fried_parameter'].tolist() == r0_a.tolist()

    def run(env):
        out = []
        for t in range(3):
            env.step(_actions(B, 40 + t))
            out.append(_outputs(env) + (env._h.get_screens(),))
        return out

    same = AOVecEnv(B, atm_fried=r0_a, **kw)
    other = AOVecEnv(B, atm_fried=r0_b, **kw)
    same.set_state(st)
    other.set_state(st)
    assert other.fried_parameter.tolist() == r0_a.tolist()
    for x, y in zip(run(same), run(other)):
        for g, w in zip(x, y):
            assert np.array_equal(g, w)
    # a state dict written before per-env strengths existed: the handle keeps its own values
    old = {k: v for k, v in st.items() if k != 'fried_parameter'}
    kept = AOVecEnv(B, atm_fried=r0_b, **kw)
    kept.set_state(old)
    assert kept.fried_parameter.tolist() == r0_b.tolist()
    ref = AOVecEnv(B, atm_fried=r0_a, **kw)
    ref.set_state(dict(old, fried_parameter=r0_b))
    for x, y in zip(run(kept), run(ref)):
        for g, w in zip(x, y):
            assert np.array_equal(g, w)
    for e in (a, same, other, kept, ref):
        e.close()


def test_more_envs_than_one_chunk_index_by_global_env():
    """env e of a 4096 + 200 env batch (two chunks) against a one-env handle with env_id_base = e: the kernels read the
    sqrt(Cn^2) of the env's position in the whole handle, not in its chunk."""
    from adaptive_optics_gym_b200 import AOVecEnv
    B = 4096 + 200
    r0 = np.where((np.arange(B) // 3) % 2 == 1, 0.20, 0.08)         # env 4096 + i and env i differ for some i
    kw = _kw('dynamic', seed=1, precision='fused')
    big = AOVecEnv(B, atm_fried=r0, **kw)
    assert big._h.chunk_size() == 4096
    probe = [0, 4, 4095, 4096, 4097, 4100, B - 1]
    assert len({r0[e] for e in probe}) == 2 and r0[4096] != r0[0]
    singles = {e: AOVecEnv(1, atm_fried=float(r0[e]), env_id_base=e, **kw) for e in probe}
    for e, s in singles.items():
        assert np.array_equal(big._h.get_screens(e, 1), s._h.get_screens()), f'construction, env {e}'
    big.reset()
    big.step(_actions(1, 0).repeat(B, 1))
    for e, s in singles.items():
        s.reset()
        s.step(_actions(1, 0))
        want = s._h.get_screens()
        np.testing.assert_allclose(big._h.get_screens(e, 1), want, rtol=0, atol=1e-12 * np.abs(want).max(),
                                   err_msg=f'after an extrusion step, env {e}')
    big.close()
    for s in singles.values():
        s.close()


def test_fallback_forms_agree_on_a_mixed_batch(monkeypatch):
    """the gathered extrusion (AOG_AR_GATHER=1) and the GEMM / complex syntheses (AOG_SCR_GEMM=1, AOG_SCR_COMPLEX=1)
    scale each env by its own sqrt(Cn^2) like the default forms (tolerances of their existing tests)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    r0 = [0.05, 0.20, 0.08, 0.10, 0.15, 0.06, 0.30]

    def extruded():
        env = AOVecEnv(7, atm_fried=r0, **_kw('dynamic', seed=5, precision='fused'))
        env.reset()
        for t in range(4):
            env.step(_actions(7, t))
        out = env._h.get_screens()
        env.close()
        return out

    def synthesised():
        env = AOVecEnv(7, atm_fried=r0, **_kw('semi_dynamic', seed=11, precision='f64'))
        env.reset()
        out = env._h.get_screens()
        env.close()
        return out

    direct, fft = extruded(), synthesised()
    monkeypatch.setenv('AOG_AR_GATHER', '1')
    gathered = extruded()
    monkeypatch.delenv('AOG_AR_GATHER')
    np.testing.assert_allclose(direct, gathered, rtol=0, atol=1e-12 * np.abs(gathered).max())
    monkeypatch.setenv('AOG_SCR_GEMM', '1')
    gemm = synthesised()
    monkeypatch.setenv('AOG_SCR_COMPLEX', '1')
    slow = synthesised()
    assert not np.array_equal(fft, gemm)
    for s in (fft, gemm):
        assert np.abs(s - slow).max() <= 1e-11 * np.abs(slow).max()
