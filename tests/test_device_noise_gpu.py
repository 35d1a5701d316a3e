"""GPU: the randomness the device draws itself against the host model of tests/test_device_noise.py.  Philox words
bit for bit; both Box-Muller generators over every 24-bit uniform; the per-episode screen synthesis against an FP64
host synthesis of the same normals; the phase tiles a synthesis writes; and extrusions with device noise against the
oracle driven by the device's own normals (read through the ``aog_debug_normals`` hook), over full turns of the
extrusion ring.  The module runs in about 40 s on one B200 (1000 W power limit)."""
import ctypes as C

import numpy as np
import pytest

from tests.test_device_noise import (PHILOX_KAT, extrusion_blocks, extrusion_normals, philox4x32_10,
                                     synthesis_blocks, synthesis_normals, uniform_f32)
from tests.test_parity_gpu import RTOL, _close, _close_obs, _mk, _screen

pytestmark = pytest.mark.gpu

KW_SMALL = dict(act_type='zernike', act_dim=6, obs_dim=2, rew_type='strehl_ratio')     # cheap host tables


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def device_philox(ctr, key, generator=0):
    """(raw words [n][4] uint32, normals [n][4] float32) of Philox blocks (counter [n][4], key [n][2]) on the device"""
    from adaptive_optics_gym_b200._lib import load
    words = np.ascontiguousarray(np.concatenate([ctr, key], axis=1), dtype=np.uint32)
    n = words.shape[0]
    raw, z = np.empty((n, 4), np.uint32), np.empty((n, 4), np.float32)
    assert load().aog_debug_normals(0, generator, 1, n, _ptr(words), _ptr(raw), _ptr(z)) == 0
    return raw, z


def device_normals(raw, generator):
    """normals [n][4] float32 the device makes of raw words [n][4]"""
    from adaptive_optics_gym_b200._lib import load
    raw = np.ascontiguousarray(raw, dtype=np.uint32)
    z = np.empty(raw.shape, np.float32)
    assert load().aog_debug_normals(0, generator, 0, raw.shape[0], _ptr(raw), None, _ptr(z)) == 0
    return z


def device_extrusion_noise(h, b, n_ext):
    """the normals [n_ext][Np] the next step's extrusions of env b of handle h draw"""
    c = h.cfg
    Np, draw0 = c.num_pupil_pixels, h.counters().extrusions
    if n_ext == 0:
        return np.zeros((0, Np))
    blocks = [extrusion_blocks(c.seed, c.env_id_base + b, draw0 + e, Np) for e in range(n_ext)]
    _, z = device_philox(np.concatenate([x[0] for x in blocks]), np.concatenate([x[1] for x in blocks]))
    z = z.reshape(n_ext, -1, 4)
    return np.stack([extrusion_normals(z[e], Np) for e in range(n_ext)]).astype(np.float64)


def host_screen(env, b, draw, sqrt_cn2):
    """FP64 host synthesis [Np^2] ([y][x]) of env b's screen at synthesis `draw`, on the device's own normals"""
    from adaptive_optics_gym_b200.tables import synthesize_screen
    c = env._h.cfg
    N, N2 = c.num_pupil_pixels, c.num_screen_fine
    _, z = device_philox(*synthesis_blocks(c.seed, c.env_id_base + b, draw, N, N2))
    z1, z2 = synthesis_normals(z, N, N2)
    return synthesize_screen(env.tables, z1, z2, sqrt_cn2)


# ------------------------------------------------------------------------------------------------ (a) Philox
@pytest.mark.parametrize('generator', [0, 1])
def test_philox_matches_host_model_bit_for_bit(generator):
    """Both copies of Philox-4x32-10 (extrusion / synthesis, camera) reproduce Random123's known answers and the host
    model on 2^20 random counters and keys; the normals of the Philox path equal those of the same words given raw."""
    raw, _ = device_philox(np.array([k[0] for k in PHILOX_KAT], np.uint32), np.array([k[1] for k in PHILOX_KAT], np.uint32),
                           generator)
    assert raw.tolist() == [k[2] for k in PHILOX_KAT]
    rng = np.random.default_rng(100 + generator)
    ctr = rng.integers(0, 2 ** 32, (1 << 20, 4), dtype=np.uint32)
    key = rng.integers(0, 2 ** 32, (1 << 20, 2), dtype=np.uint32)
    raw, z = device_philox(ctr, key, generator)
    assert np.array_equal(raw, philox4x32_10(ctr, key))
    assert np.array_equal(z.view(np.uint32), device_normals(raw, generator).view(np.uint32))


# ------------------------------------------------------------------------------------------------ (b) Box-Muller
# Error model of the FP32 Box-Muller z = r cos t, r sin t (r = sqrt(-2 ln u), t = 2 pi u') against FP64 on the same u.
# CUDA C Programming Guide, intrinsic functions: __logf has an absolute error of at most 2^-21.41 on [0.5, 2] and 3 ulp
# elsewhere; __sinf / __cosf 2^-21.41 absolute on [-pi, pi].
A_SFU = 2.0 ** -21.41
# angle: 2 pi u rounded to FP32 with the FP32 constant 6.28318530718f (2 pi (2^-24 + 2.8e-8) <= 0.55e-6), the scaling
# into revolutions ahead of MUFU.SIN / COS (2 pi 2^-23 = 0.75e-6), the SFU's own 2^-21.41 (0.36e-6): 1.7e-6 -> 2e-6
ANGLE_ERR = 2e-6
# The top of the range, u >= 1 - 2^-20 (radius below 1.4e-3), has its own looser bound: there the radicand's absolute
# error dominates, |r' - r| <= sqrt(2 x 2^-21.41) = 8.5e-4 however small r is (u = 1.0 itself has r = 0).
TOP = 1.0 - 2.0 ** -20
TOP_BOUND = 9e-4


def normal_error_bound(u):
    """Bound on |z_device - z_fp64| at radius uniform u (FP64 array): an error d of ln u moves r^2 by 2 d, so r by at
    most min(2 d / r, sqrt(2 d)); sqrt (IEEE or sqrt.approx) adds 2^-22 r; the angle and the final product r x (cos or
    sin) add r (ANGLE_ERR + 2^-23).  d = 2^-21.41 + 2^-21 |ln u| covers both of __logf's regimes."""
    L = -np.log(u)
    r = np.sqrt(2.0 * L)
    d = A_SFU + 2.0 ** -21 * L
    with np.errstate(divide='ignore'):
        dr = np.minimum(np.sqrt(2.0 * d), 2.0 * d / r)
    return dr + r * (2.0 ** -22 + ANGLE_ERR + 2.0 ** -23)


@pytest.mark.parametrize('generator', [0, 1])
def test_box_muller_every_uniform(generator):
    """Raw words k << 8 in all four lanes for every k < 2^24: every radius and angle uniform occurs.  Every normal is
    finite, |z| <= 5.9, within normal_error_bound (TOP_BOUND at the top of the range) of the FP64 Box-Muller, and lanes
    2, 3 repeat lanes 0, 1."""
    assert normal_error_bound(np.array([TOP]))[0] <= TOP_BOUND
    worst, worst_top, worst_ratio = 0.0, 0.0, 0.0
    chunk = 1 << 22
    for k0 in range(0, 1 << 24, chunk):
        k = np.arange(k0, k0 + chunk, dtype=np.uint32) << np.uint32(8)
        z = device_normals(np.repeat(k[:, None], 4, axis=1), generator)
        assert np.all(np.isfinite(z)), f'non-finite normal at k = {k0 + np.flatnonzero(~np.isfinite(z).all(1))[:8]}'
        assert np.array_equal(z[:, 2:].view(np.uint32), z[:, :2].view(np.uint32))
        assert np.abs(z).max() <= 5.9
        u = uniform_f32(k).astype(np.float64)
        r, t = np.sqrt(-2.0 * np.log(u)), 2.0 * np.pi * u
        err = np.maximum(np.abs(z[:, 0] - r * np.cos(t)), np.abs(z[:, 1] - r * np.sin(t)))
        top = u >= TOP
        bound = np.where(top, TOP_BOUND, normal_error_bound(u))
        bad = err > bound
        assert not bad.any(), f'generator {generator}: error {err[bad][:4]} > {bound[bad][:4]} at u = {u[bad][:4]}'
        worst = max(worst, float(err[~top].max()))
        worst_top = max(worst_top, float(err[top].max()) if top.any() else 0.0)
        worst_ratio = max(worst_ratio, float((err / bound).max()))
    print(f'\n[box-muller] generator {generator}: max |z - z_fp64| {worst:.3e} for u < 1 - 2^-20, '
          f'{worst_top:.3e} for u >= 1 - 2^-20; largest error / bound {worst_ratio:.3f}')


# ------------------------------------------------------------------------------------------------ (c) synthesis
def _check_screens(env, envs, draw, sqrt_cn2, what):
    for b in envs:
        got = env._h.get_screens(b, 1)[0]
        want = host_screen(env, b, draw, sqrt_cn2[b])
        err = np.abs(got - want).max()
        assert err <= 1e-11 * np.abs(want).max(), f'{what}: env {b} differs from the host synthesis by {err:.3e}'


@pytest.mark.parametrize('form', ['fft', 'gemm', 'complex'])
def test_screen_synthesis_matches_host_fp64(form, monkeypatch):
    """Construction, two consecutive resets (screen_draws advances), reset(seed=), with env_id_base = 3 and a Fried
    parameter per env, in each synthesis form: the 240-point FFT (default), the real tensor-core GEMMs
    (AOG_SCR_GEMM=1) and the complex GEMMs (AOG_SCR_COMPLEX=1)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    from adaptive_optics_gym_b200.tables import sqrt_cn2_from_fried
    if form != 'fft':
        monkeypatch.setenv('AOG_SCR_GEMM', '1')
    if form == 'complex':
        monkeypatch.setenv('AOG_SCR_COMPLEX', '1')
    r0 = [0.08, 0.15, 0.30, 0.05, 0.12]
    env = AOVecEnv(5, atm_type='semi_dynamic', atm_fried=r0, seed=21, env_id_base=3, precision='f64', **KW_SMALL)
    sq = sqrt_cn2_from_fried(r0, env.wavelength_sci)
    envs = range(5)
    assert env._h.counters().screen_draws == 1
    _check_screens(env, envs, 0, sq, 'construction')
    for draw in (1, 2):
        env.reset()
        assert env._h.counters().screen_draws == draw + 1
        _check_screens(env, envs, draw, sq, f'reset {draw}')
    env.reset(seed=99)
    assert env._h.counters().screen_draws == 1 and env._h.cfg.seed == 99
    _check_screens(env, envs, 0, sq, 'reset(seed=99)')
    env.close()


def test_screen_synthesis_128_pupil_matches_host_fp64():
    """A 128^2 pupil: the real-arithmetic GEMM form (the FFT form is for 240^2 only)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    env = AOVecEnv(3, atm_type='semi_dynamic', atm_fried=0.15, seed=4, num_pupil_pixels=128, num_focal_pixels_fiber=64,
                   precision='f64', **KW_SMALL)
    sq = [float(np.sqrt(env.tables['cn2']))] * 3
    _check_screens(env, range(3), 0, sq, 'construction')
    env.reset()
    _check_screens(env, range(3), 1, sq, 'reset')
    env.close()


def test_screen_synthesis_beyond_one_chunk_matches_host_fp64():
    """4096 + 40 envs: the second chunk keys its envs by their global id (envs 4096 and 4135)."""
    from adaptive_optics_gym_b200 import AOVecEnv
    B = 4096 + 40
    env = AOVecEnv(B, atm_type='semi_dynamic', atm_fried=0.15, seed=8, precision='fused', **KW_SMALL)
    assert env._h.chunk_size() == 4096
    sq = [float(np.sqrt(env.tables['cn2']))] * B
    _check_screens(env, (0, 4095, 4096, 4135), 0, sq, 'construction')
    env.reset()
    _check_screens(env, (0, 4095, 4096, 4135), 1, sq, 'reset')
    env.close()


# ------------------------------------------------------------------------------------------------ (d) phase tiles


@pytest.mark.parametrize('form', ['fft', 'gemm'])
@pytest.mark.parametrize('precision', ['fused', 'tensor'])
def test_phase_tiles_written_by_the_synthesis(precision, form, monkeypatch):
    """The fixed-point phase tiles the synthesis writes (k_scr_combine4 after the FFT form, the tile refresh after
    the GEMM form): a reset and two steps of a 12-env batch (tcgen05 kernels) against the oracle on the screens read
    back, envs 0 and 11."""
    import torch
    from adaptive_optics_gym_b200 import AOVecEnv
    from oracle.ao_oracle import OracleAOEnv
    if form == 'gemm':
        monkeypatch.setenv('AOG_SCR_GEMM', '1')
    B = 12
    kw = dict(KW_SMALL, atm_fried=0.15, timesteps_per_episode=3)
    env = AOVecEnv(B, atm_type='semi_dynamic', seed=31, precision=precision, **kw)
    env.reset()                                             # a device synthesis (the second draw) and its tiles
    screens = env._h.get_screens()
    rng = np.random.default_rng(5)
    acts = rng.uniform(-1, 1, (2, B, 6)).astype(np.float32)
    outs = [(env.obs_f64.cpu().numpy().copy(), None, None)]
    for t in range(2):
        _, rew, _, _, info = env.step(torch.from_numpy(acts[t]).cuda())
        torch.cuda.synchronize()
        outs.append((env.obs_f64.cpu().numpy().copy(), rew.cpu().numpy().copy(), info['power'].cpu().numpy().copy()))
    env.close()
    ref = OracleAOEnv(atm_type='quasi_static', **kw, initial_screen=screens[0])
    for b in (0, B - 1):
        ref.layer.achromatic_screen = screens[b].copy()
        ref.reset()
        _close_obs(outs[0][0][b], ref.last_obs_f64, f'env {b} reset obs')
        for t in range(2):
            _, rr, _, _, rinfo = ref.step(acts[t][b])
            _close_obs(outs[t + 1][0][b], ref.last_obs_f64, f'env {b} obs step {t}')
            _close(outs[t + 1][1][b], rr, 1e-5, f'env {b} reward step {t}')
            _close(outs[t + 1][2][b], rinfo['power'], 1e-5, f'env {b} power step {t}')


# ------------------------------------------------------------------------------------------------ (e) extrusion
KW_DYN = dict(KW_SMALL, atm_type='dynamic', atm_fried=0.10, timesteps_per_episode=10)


def _oracle_and_tables(vel, seed, sh=False, **kw):
    from oracle.ao_oracle import OracleAOEnv
    scr = _screen(seed, 0.10)
    ref = OracleAOEnv(**dict(KW_DYN, **kw), atm_vel=vel, initial_screen=scr, seed=seed, SH_operation=sh)
    lay = ref.layer
    tabs = dict(ar_stencil=np.flatnonzero(lay.stencil_left).astype(np.int32), ar_A=lay.A_horizontal,
                ar_B=lay.B_horizontal)
    if sh:
        s = ref.shwfs
        idx = s.estimation_subapertures
        tabs.update(sh_recon=ref.reconstruction_matrix, sh_offset=np.array((s.mla_x[idx], s.mla_y[idx])) + ref.slopes_ref)
    return ref, scr, tabs


def _step_against_oracle(env, ref, a, rtol, what, ra=None):
    """one step of env with its device noise and of the oracle with the same normals; -> (extrusions, wrapped, done)"""
    n_ext = ref.num_extrusions_for_next_step()
    assert env._h.next_extrusions() == n_ext, what
    noise = device_extrusion_noise(env._h, 0, n_ext)
    org = env._h.counters().column_origin
    o, r, d, _, info = env.step(a)
    ro, rr, rd, _, rinfo = ref.step(a if ra is None else ra, extrusion_noise=noise)
    org2 = env._h.counters().column_origin
    assert d == rd, what
    S = ref.layer.achromatic_screen
    err = np.abs(env._h.get_field('screen') - S).max()
    assert err <= 1e-9 * np.abs(S).max(), f'{what}: screen error {err:.3e} of max {np.abs(S).max():.3e}'
    if rtol >= 1e-5:          # tensor / fused: the detector powers' amplitude floor of _close_obs
        _close_obs(env.last_obs_f64, ref.last_obs_f64, f'{what} obs')
    else:
        _close(env.last_obs_f64, ref.last_obs_f64, max(rtol, 1e-7), f'{what} obs')
    _close(r, rr, max(rtol, 1e-7), f'{what} reward')
    _close(info['power'], rinfo['power'], max(rtol, 1e-7), f'{what} power')
    wrapped = (org2 < org) if ref.velocity > 0 else (org2 > org)
    return n_ext, wrapped and n_ext > 0, d


@pytest.mark.parametrize('precision,vel,steps,gathered', [
    ('f64', 20, 27, False), ('f64', -20, 27, False), ('tensor', 20, 27, False), ('tensor', -20, 27, False),
    ('fused', 20, 27, False), ('fused', -20, 27, False), ('f64', -20, 27, True), ('fused', 1, 12, False)])
def test_extrusion_device_noise_against_oracle(precision, vel, steps, gathered, monkeypatch):
    """Device Philox extrusion noise, fetched through the hook and fed to the oracle: the screen after every step
    agrees to 1e-9 of its maximum and the outputs at the injected-noise tolerances.  27 steps of +-20 m/s (9.6 px per
    step) pass more than a full turn of the 240-column ring, with episode boundaries at steps 10 and 20; 1 m/s
    (0.48 px per step) has steps without extrusions; AOG_AR_GATHER=1 is the gathered form.  Then get_state, set_state
    into a fresh handle, which continues equal to the oracle."""
    if gathered:
        monkeypatch.setenv('AOG_AR_GATHER', '1')
    ref, scr, tabs = _oracle_and_tables(vel, 40 + steps + (vel > 0))
    kw = dict(KW_DYN, atm_vel=vel, initial_screen=scr, tables=tabs, seed=2 ** 40 + 7)
    env = _mk(precision, **kw)
    rtol = RTOL[precision]
    rng = np.random.default_rng(abs(vel))
    env.reset(), ref.reset()
    total, wraps, zero_steps = 0, 0, 0
    for t in range(steps):
        n, w, d = _step_against_oracle(env, ref, rng.uniform(-1, 1, 6).astype(np.float32), rtol, f'step {t}')
        total, wraps, zero_steps = total + n, wraps + w, zero_steps + (n == 0)
        if d:
            env.reset(), ref.reset()
            _close(env.last_obs_f64, ref.last_obs_f64, max(rtol, 1e-7), f'reset after step {t}')
    assert env._h.counters().extrusions == total
    if abs(vel) == 20:
        assert total > 240 and wraps >= 1
    else:
        assert zero_steps > 0 and total > 0
    st = env.get_state()
    env.close()
    env = _mk(precision, **kw)
    env.set_state(st)
    for t in range(3):
        _step_against_oracle(env, ref, rng.uniform(-1, 1, 6).astype(np.float32), rtol, f'after set_state step {t}')
    env.close()


def test_extrusion_device_noise_shack_hartmann_closed_loop():
    """SH_step (noise-free camera) then step with its action, device extrusion noise, through one turn of the ring,
    against the oracle at the tolerances of test_config4_shack_hartmann_closed_loop (FP64 handle)."""
    ref, scr, tabs = _oracle_and_tables(20, 77, sh=True)
    env = _mk('f64', **KW_DYN, atm_vel=20, initial_screen=scr, tables=tabs, seed=12345, SH_operation=True)
    env.reset(), ref.reset()
    total, wraps = 0, 0
    for t in range(26):
        a, _ = env.SH_step(noise='none')
        ra = np.array(ref.SH_step(poisson=False)[0])
        np.testing.assert_allclose(a, ra, rtol=0, atol=1e-8 * np.abs(ra).max())
        n, w, d = _step_against_oracle(env, ref, a, 1e-6, f'step {t}', ra=ra)
        total, wraps = total + n, wraps + w
        if d:
            env.reset(), ref.reset()
    assert total > 240 and wraps >= 1
    env.close()


# ------------------------------------------------------------------------------------------------ (f) per-env keys
def test_extrusion_per_env_keys_in_a_batch():
    """130 envs (two 112-env extrusion tiles, five 32-env tile groups), env_id_base = 5, a Fried parameter per env,
    device noise: envs 0, 111, 112 and 129 against oracles fed each env's own normals, for a full turn of the ring."""
    import torch
    from adaptive_optics_gym_b200 import AOVecEnv
    from oracle.ao_oracle import OracleAOEnv
    B, R, steps = 130, 3, 26
    r0 = [(0.08, 0.10, 0.14, 0.20, 0.12)[b % 5] for b in range(B)]
    ref0, _, tabs = _oracle_and_tables(20, 90)
    scr = [_screen(91 + i, 0.10) for i in range(R)]
    env = AOVecEnv(B, **dict(KW_DYN, atm_fried=r0), atm_vel=20, initial_screens=np.stack([scr[b % R] for b in range(B)]),
                   tables=tabs, seed=3, env_id_base=5, precision='fused')
    check = (0, 111, 112, 129)
    refs = {b: OracleAOEnv(**dict(KW_DYN, atm_fried=r0[b]), atm_vel=20, initial_screen=scr[b % R], seed=90)
            for b in check}
    for ref in refs.values():
        assert np.array_equal(ref.layer.stencil_left, ref0.layer.stencil_left)
        ref.reset()
    env.reset()
    rng = np.random.default_rng(9)
    total = 0
    for t in range(steps):
        n_ext = env._h.next_extrusions()
        noise = {b: device_extrusion_noise(env._h, b, n_ext) for b in check}
        a = rng.uniform(-1, 1, (B, 6)).astype(np.float32)
        _, rew, done, _, info = env.step(torch.from_numpy(a).cuda())
        torch.cuda.synchronize()
        total += n_ext
        for b, ref in refs.items():
            assert ref.num_extrusions_for_next_step() == n_ext
            _, rr, rd, _, rinfo = ref.step(a[b], extrusion_noise=noise[b])
            S = ref.layer.achromatic_screen
            err = np.abs(env._h.get_screens(b, 1)[0] - S).max()
            assert err <= 1e-9 * np.abs(S).max(), f'env {b} step {t}: screen error {err:.3e}'
            _close_obs(env.obs_f64[b].cpu().numpy(), ref.last_obs_f64, f'env {b} step {t} obs')
            _close(rew[b].item(), rr, 1e-5, f'env {b} step {t} reward')
            _close(info['power'][b].item(), rinfo['power'], 1e-5, f'env {b} step {t} power')
            assert bool(done[b]) == rd
        if bool(done[0]):
            env.reset()
            for ref in refs.values():
                ref.reset()
    assert total > 240
    env.close()
