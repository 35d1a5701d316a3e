"""The fused tcgen05 optics kernel at a 512^2 pupil (BASELINE configs[4], the largest point of the pupil-grid axis).
k_dm_phase_tc runs every pupil column as two 256-pixel MMA segments there; these tests hold it to the CPU oracle and
to the FP64 path.  Tolerances as in test_parity_gpu.py: 1e-5 relative, detector pixels plus the amplitude floor of
the fixed-point phase and the SFU's sin / cos (``_close_obs``)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NP = 512


def _screen(seed, r0=0.15, n=NP):
    from oracle.ao_oracle import hcipy_make_pupil_grid, hcipy_Cn_squared_from_fried_parameter, von_karman_screen
    g = hcipy_make_pupil_grid(n, 0.5)
    cn2 = hcipy_Cn_squared_from_fried_parameter(r0, 2.2e-6)
    return von_karman_screen(g, cn2, 10.0, np.random.default_rng(seed))


def _close_obs(got, want, what, amp_floor=1e-8):
    """Detector powers against FP64: 1e-5 relative plus an absolute amplitude error of up to ``amp_floor`` of the peak
    amplitude (tools/dark_pixel_error_model.py), i.e. a power error of 2 amp_floor sqrt(P P_max)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    peak = want.max(axis=-1, keepdims=True)
    tol = 1e-5 * want + 2 * amp_floor * np.sqrt(want * peak)
    bad = np.abs(got - want) > tol
    assert not bad.any(), f'{what}: {np.abs(got - want)[bad]} > {tol[bad]} at brightness {(want / peak)[bad]}'


def _close(a, b, rtol, what):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    assert np.all(err <= rtol), f'{what}: max rel err {err.max():.3e} > {rtol} (got {a}, want {b})'


CASES = [(128, 2, 'num_actuators', 64, 'strehl_ratio'), (256, 5, 'zernike', 6, 'smf_ssim')]


@pytest.mark.parametrize('Nf,obs_dim,act_type,K,rew_type', CASES)
def test_pupil512_fused_against_oracle(Nf, obs_dim, act_type, K, rew_type):
    """Quasi-static, 3 steps, against OracleAOEnv built at the same grid.  A single env (B = 1: batches of up to 8 run
    the tensor-core kernel at 512^2) and a 3-env batch whose env 0 must equal the single env bit for bit."""
    import torch
    from adaptive_optics_gym_b200 import AOEnv, AOVecEnv
    from oracle.ao_oracle import OracleAOEnv
    kw = dict(atm_type='quasi_static', atm_fried=0.15, act_type=act_type, act_dim=K, obs_dim=obs_dim, rew_type=rew_type,
              timesteps_per_episode=3, num_pupil_pixels=NP, num_focal_pixels_fiber=Nf)
    scr = np.stack([_screen(NP + Nf + i) for i in range(3)])
    env = AOEnv(**kw, precision='fused', initial_screen=scr[0])
    vec = AOVecEnv(3, **kw, precision='fused', initial_screens=scr)
    ref = OracleAOEnv(**kw, initial_screen=scr[0])
    rng = np.random.default_rng(Nf)
    env.reset(), ref.reset(), vec.reset()
    _close_obs(env.last_obs_f64, ref.last_obs_f64, 'reset obs')
    for t in range(3):
        a = rng.normal(0, 0.7, (3, K)).astype(np.float32)
        o, r, d, _, info = env.step(a[0])
        ro, rr, rd, _, rinfo = ref.step(a[0])
        vo, vr, vd, _, vinfo = vec.step(torch.from_numpy(a).cuda())
        torch.cuda.synchronize()
        assert d == rd == bool(vd[0])
        _close_obs(env.last_obs_f64, ref.last_obs_f64, f'obs step {t}')
        _close(r, rr, 1e-5, 'reward')
        _close(info['power'], rinfo['power'], 1e-5, 'power')
        assert vr[0].item() == r and vinfo['power'][0].item() == info['power']
        assert np.array_equal(vo[0].cpu().numpy().view(np.uint16), o.view(np.uint16))
        assert np.array_equal(vec.obs_f64[0].cpu().numpy(), env.last_obs_f64)
    env.close(), vec.close()


def test_pupil512_generic_table_kernel_against_oracle(monkeypatch):
    """AOG_FUSED_GENERIC=1: the kernel variant for tables without the conjugate-pair symmetry (kernel MODE 1)."""
    monkeypatch.setenv('AOG_FUSED_GENERIC', '1')
    test_pupil512_fused_against_oracle(*CASES[0])


def test_pupil512_full_batch_properties():
    """4096 envs at 512^2 (32 env blocks of 1024 column segments, 2^30 pupil pixels in all): env i carries screen and
    action i % 8, so all 512 copies of a case must agree, and the 8 cases must agree with an 8-env FP64 run (1e-5).
    Detector pixels: a 2x2 detector at r0 = 0.20 m has speckle pixels near 1e-4 of the brightest one, where the
    amplitude floor decides.  Its largest source is the tensor cores' truncating FP32 accumulation of the DM phase, an
    error with the sign and smoothness of the DM surface that adds up coherently over the pupil:
    ``python tools/dark_pixel_error_model.py --pupil 512 --r0 0.20 --obs-dim 2`` bounds it by 1.3e-7 ... 5.4e-7 of the
    peak amplitude (measured here: 8.7e-8 on a pixel at 1.7e-4 of the brightest, 1.3e-5 relative), hence 6e-7."""
    import torch
    from adaptive_optics_gym_b200 import AOVecEnv
    B, R = 4096, 8
    kw = dict(atm_fried=0.20, act_dim=64, obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=4,
              num_pupil_pixels=NP)
    scr = np.stack([_screen(60 + i, r0=0.20) for i in range(R)]).astype(np.float32)
    scr[0] = 0.0                                                   # case 0: flat wavefront
    rng = np.random.default_rng(9)
    acts = rng.uniform(-1, 1, (3, R, 64)).astype(np.float32)
    big = AOVecEnv(B, **kw, initial_screens=np.tile(scr, (B // R, 1)), precision='fused')
    ref = AOVecEnv(R, **kw, initial_screens=scr, precision='f64')
    big.reset(), ref.reset()
    for t in range(3):
        obs, rew, done, _, info = big.step(torch.from_numpy(np.tile(acts[t], (B // R, 1))).cuda())
        o_r, r_r, _, _, i_r = ref.step(torch.from_numpy(acts[t]).cuda())
        torch.cuda.synchronize()
        o64 = big.obs_f64.reshape(B // R, R, 4)
        for x in (o64, rew.reshape(-1, R), info['power'].reshape(-1, R), big.strehl.reshape(-1, R)):
            x0 = x[:1].expand_as(x)
            assert torch.all((x - x0).abs() <= 1e-12 * x0.abs()), f'copies of one case differ (step {t})'
        _close_obs(o64[0].cpu().numpy(), ref.obs_f64.cpu().numpy(), f'obs step {t}', amp_floor=6e-7)
        _close(rew[:R].cpu().numpy(), ref.reward.cpu().numpy(), 1e-5, f'reward step {t}')
        _close(info['power'][:R].cpu().numpy(), i_r['power'].cpu().numpy(), 1e-5, f'power step {t}')
        _close(big.strehl[:R].cpu().numpy(), ref.strehl.cpu().numpy(), 1e-5, f'strehl step {t}')
    big.close(), ref.close()


def test_pupil512_dynamic_extrusion_injected_noise():
    """dynamic, v = 20 m/s with the oracle's AR tables and injected extrusion noise: the extrusion epilogue refreshes
    the 512^2 phase tiles every step; obs, reward and power against OracleAOEnv."""
    from adaptive_optics_gym_b200 import AOEnv
    from oracle.ao_oracle import OracleAOEnv
    kw = dict(atm_type='dynamic', atm_vel=20, atm_fried=0.10, act_dim=64, obs_dim=2, rew_type='strehl_ratio',
              timesteps_per_episode=3, num_pupil_pixels=NP)
    scr = _screen(7, 0.10)
    ref = OracleAOEnv(**kw, initial_screen=scr, seed=11)
    lay = ref.layer
    tabs = dict(ar_stencil=np.flatnonzero(lay.stencil_left).astype(np.int32), ar_A=lay.A_horizontal,
                ar_B=lay.B_horizontal)
    env = AOEnv(**kw, precision='fused', initial_screen=scr, tables=tabs)
    rng = np.random.default_rng(8)
    total_ext = 0
    env.reset(), ref.reset()
    _close_obs(env.last_obs_f64, ref.last_obs_f64, 'reset obs')
    for t in range(3):
        n_ext = ref.num_extrusions_for_next_step()
        assert env._h.next_extrusions() == n_ext
        total_ext += n_ext
        noise = rng.standard_normal((n_ext, NP))
        a = rng.uniform(-1, 1, 64).astype(np.float32)
        o, r, d, _, info = env.step(a, extrusion_noise=noise)
        ro, rr, rd, _, rinfo = ref.step(a, extrusion_noise=noise)
        assert d == rd
        _close_obs(env.last_obs_f64, ref.last_obs_f64, f'obs step {t}')
        _close(r, rr, 1e-5, 'reward')
        _close(info['power'], rinfo['power'], 1e-5, 'power')
    assert total_ext > 0 and env._h.counters().extrusions == total_ext
    env.close()
