"""CPU: a host model of the random streams the device draws itself -- Philox-4x32-10, the FP32 uniform, an FP64
Box-Muller, and the counter / key maps of the extrusion noise and of the screen synthesis -- checked against known
answers.  tests/test_device_noise_gpu.py compares the device with this model through the ``aog_debug_normals`` hook."""
import numpy as np
import pytest

MASK32 = np.uint64(0xFFFFFFFF)
SYNTH_KEY_XOR = 0x9E3779B97F4A7C15          # aog_generate_screens: the synthesis key is the seed XOR this constant


def philox4x32_10(counter, key):
    """Philox-4x32-10 (Salmon et al. 2011) in uint64 arithmetic: counter [..., 4], key [..., 2] uint32 words ->
    [..., 4] uint32, the rounds of aog_philox4x32_10 (csrc/kernels_f64.cuh)."""
    c = np.asarray(counter, dtype=np.uint64)
    k = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (c[..., i].copy() for i in range(4))
    k0, k1 = k[..., 0].copy(), k[..., 1].copy()
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0            # both factors < 2^32: the product is exact in 64 bits
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK32
        k0 = (k0 + np.uint64(0x9E3779B9)) & MASK32
        k1 = (k1 + np.uint64(0xBB67AE85)) & MASK32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def uniform_f32(words):
    """The device's uniform of a 32-bit word, formed in FP32 as it is: ((float)(r >> 8) + 0.5f) * 2^-24.  Above 2^23
    the sum rounds to even, so the top words give 1 - 2^-23 and exactly 1.0."""
    r = np.asarray(words, dtype=np.uint32)
    return ((r >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def box_muller_f64(raw):
    """The four normals of raw blocks [..., 4] in FP64 from the FP32 uniforms: (r cos t, r sin t) of words (0, 1) and
    of words (2, 3), r = sqrt(-2 ln u), t = 2 pi u'."""
    u = uniform_f32(raw).astype(np.float64)
    ra, rb = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    ta, tb = 2.0 * np.pi * u[..., 1], 2.0 * np.pi * u[..., 3]
    return np.stack([ra * np.cos(ta), ra * np.sin(ta), rb * np.cos(tb), rb * np.sin(tb)], axis=-1)


def _words64(x):
    x = np.asarray(x, dtype=np.uint64)
    return x & MASK32, x >> np.uint64(32)


def extrusion_blocks(seed, env_id, draw, num_pixels):
    """Counter and key blocks of extrusion ``draw`` (the env's extrusion counter + e for the e-th extrusion of a step) of
    global env ``env_id`` (k_ar_noise / k_ar_gather): block j = (j, draw lo, draw hi, env id lo), key (seed lo,
    seed hi ^ env id hi); block j makes the normals of pixels 4 j .. 4 j + 3 of the new column."""
    nb = (num_pixels + 3) // 4
    d_lo, d_hi = _words64(draw)
    e_lo, e_hi = _words64(env_id)
    s_lo, s_hi = _words64(seed)
    ctr = np.stack([np.arange(nb, dtype=np.uint64), np.full(nb, d_lo), np.full(nb, d_hi), np.full(nb, e_lo)], axis=-1)
    key = np.tile(np.array([s_lo, s_hi ^ e_hi], dtype=np.uint64), (nb, 1))
    return ctr.astype(np.uint32), key.astype(np.uint32)


def extrusion_normals(z, num_pixels):
    """Normals [num_pixels] of one extrusion from the normals [nb][4] of its blocks (pixel i = lane i % 4 of block i / 4)."""
    return np.asarray(z).reshape(-1)[:num_pixels]


def synthesis_blocks(seed, env_id, screen_draw, n, n2):
    """Counter and key blocks of synthesis ``screen_draw`` (the handle's screen_draws counter before it) of global env
    ``env_id`` (k_scr_fft_rows / k_scr_noise_planes / k_scr_noise): element i of the fine scale's n x n spectrum and
    element i of the coarse scale's n2 x n2 one (at offset n^2) are drawn at pair = (screen_draw (n^2 + n2^2) + i) / 2;
    block = (pair lo, pair hi, env id lo, env id hi), key = seed ^ 0x9E3779B97F4A7C15.  Fine-scale blocks first."""
    P, Q = n * n, n2 * n2
    base = screen_draw * (P + Q)
    pairs = np.concatenate([base // 2 + np.arange(P // 2, dtype=np.uint64),
                            (base + P) // 2 + np.arange(Q // 2, dtype=np.uint64)]).astype(np.uint64)
    p_lo, p_hi = _words64(pairs)
    e_lo, e_hi = _words64(env_id)
    ctr = np.stack([p_lo, p_hi, np.full(pairs.size, e_lo), np.full(pairs.size, e_hi)], axis=-1)
    k_lo, k_hi = _words64(int(seed) ^ SYNTH_KEY_XOR)
    key = np.tile(np.array([k_lo, k_hi], dtype=np.uint64), (pairs.size, 1))
    return ctr.astype(np.uint32), key.astype(np.uint32)


def synthesis_normals(z, n, n2):
    """Complex spectral normals (z1 [n][n], z2 [n2][n2], indexed [ky][kx]) from the normals [nb][4] of the blocks of
    ``synthesis_blocks``: block j of a scale makes element 2 j = z[j][0] + i z[j][1] and 2 j + 1 = z[j][2] + i z[j][3]."""
    z = np.asarray(z, dtype=np.float64).reshape(-1, 2)
    c = z[:, 0] + 1j * z[:, 1]
    return c[:n * n].reshape(n, n), c[n * n:].reshape(n2, n2)


# ---------------------------------------------------------------------------------------------------------- tests
# Random123 known answers for Philox-4x32-10 (kat_vectors): (counter, key, result)
PHILOX_KAT = [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
]


def test_philox_known_answers():
    for ctr, key, want in PHILOX_KAT:
        assert philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32)).tolist() == want
    ctr = np.array([k[0] for k in PHILOX_KAT], np.uint32)        # vectorised: the same answers row by row
    key = np.array([k[1] for k in PHILOX_KAT], np.uint32)
    assert philox4x32_10(ctr, key).tolist() == [k[2] for k in PHILOX_KAT]


def test_uniform_rounds_to_one_at_the_top():
    top = 1 << 24
    u = uniform_f32(np.array([(top - 1) << 8, (top - 2) << 8, (top - 3) << 8, (top - 4) << 8, 0xffffffff], np.uint32))
    assert u.dtype == np.float32
    assert u[0] == np.float32(1.0) and u[4] == np.float32(1.0)         # the low 8 bits are dropped
    assert u[1] == u[2] == np.float32(1.0 - 2.0 ** -23)
    assert u[3] == np.float32(1.0 - 4 * 2.0 ** -24)                    # k + 0.5 rounds to the even neighbour k
    # below 2^23 the sum is exact: u = (k + 0.5) 2^-24, strictly inside (0, 1)
    k = np.array([0, 1, 12345, (1 << 23) - 1], np.uint32)
    assert np.array_equal(uniform_f32(k << np.uint32(8)).astype(np.float64), (k + 0.5) * 2.0 ** -24)


def test_box_muller_model():
    top = (1 << 24) - 1
    z = box_muller_f64(np.array([[top << 8, 0, top << 8, 0]], np.uint32))
    assert np.array_equal(z, np.zeros((1, 4)))                          # u = 1.0: radius 0
    z = box_muller_f64(np.array([[0, 0, 0, 1 << 30]], np.uint32))        # u = 2^-25: the largest radius
    r = np.sqrt(50 * np.log(2.0))
    assert abs(z[0, 0] - r * np.cos(2 * np.pi * 2.0 ** -25)) < 1e-15 * r and abs(z[0, 2] - r * np.cos(np.pi / 2 + 2 * np.pi * 2.0 ** -25)) < 1e-14
    assert r < 5.9
    # Philox normals of a stream are standard normal (a wrong lane or word order would not change this, but a wrong
    # uniform or radius would)
    rng = np.random.default_rng(0)
    raw = philox4x32_10(rng.integers(0, 2 ** 32, (200000, 4), dtype=np.uint32),
                        rng.integers(0, 2 ** 32, (200000, 2), dtype=np.uint32))
    z = box_muller_f64(raw).ravel()
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1) < 1e-2 and abs(np.mean(z ** 4) - 3) < 5e-2


def test_extrusion_stream_map():
    seed, env, draw = 0x0123456789ABCDEF, (7 << 32) | 0x55, (3 << 32) | 9
    ctr, key = extrusion_blocks(seed, env, draw, 240)
    assert ctr.shape == (60, 4) and key.shape == (60, 2)
    assert ctr[5].tolist() == [5, 9, 3, 0x55]
    assert key[5].tolist() == [0x89ABCDEF, 0x01234567 ^ 7]
    ctr, _ = extrusion_blocks(seed, env, draw, 241)                     # a ragged column: one more block
    assert ctr.shape == (61, 4)
    z = np.arange(61 * 4).reshape(61, 4)
    assert extrusion_normals(z, 241).tolist() == list(range(241))


def test_synthesis_stream_map():
    n, n2 = 240, 48
    seed, env = 0x0123456789ABCDEF, (2 << 32) | 17
    ctr, key = synthesis_blocks(seed, env, 0, n, n2)
    assert ctr.shape == (n * n // 2 + n2 * n2 // 2, 4)
    assert ctr[0].tolist() == [0, 0, 17, 2] and ctr[-1].tolist() == [(n * n + n2 * n2) // 2 - 1, 0, 17, 2]
    k = seed ^ SYNTH_KEY_XOR
    assert key[0].tolist() == [k & 0xFFFFFFFF, k >> 32]
    # consecutive draws take consecutive, disjoint pair ranges; a large draw index reaches the counter's high word
    c1, _ = synthesis_blocks(seed, env, 1, n, n2)
    assert c1[0, 0] == ctr[-1, 0] + 1
    big, _ = synthesis_blocks(seed, env, 1 << 20, n, n2)
    pair0 = (1 << 20) * (n * n + n2 * n2) // 2
    assert big[0].tolist() == [pair0 & 0xFFFFFFFF, pair0 >> 32, 17, 2]
    z = np.arange(ctr.shape[0] * 4, dtype=np.float64).reshape(-1, 4)
    z1, z2 = synthesis_normals(z, n, n2)
    assert z1[0, 0] == 0 + 1j and z1[0, 1] == 2 + 3j and z1[1, 0] == 2 * n + (2 * n + 1) * 1j
    assert z2[0, 0] == n * n * 2 + (n * n * 2 + 1) * 1j


def test_host_synthesis_equals_synthesize_screens():
    """``synthesize_screen`` with given normals is ``synthesize_screens`` with drawn ones (the device reference)."""
    from adaptive_optics_gym_b200.tables import screen_synthesis_tables, synthesize_screen, synthesize_screens
    tabs = screen_synthesis_tables(64, 0.5 / 64, 10.0)
    cn2 = 3.7e-13
    a = synthesize_screens(tabs, 2, cn2, np.random.default_rng(5))
    rng = np.random.default_rng(5)
    for i in range(2):
        z1 = rng.standard_normal((64, 64)) + 1j * rng.standard_normal((64, 64))
        z2 = rng.standard_normal((48, 48)) + 1j * rng.standard_normal((48, 48))
        assert np.array_equal(a[i], synthesize_screen(tabs, z1, z2, np.sqrt(cn2)))
    # the FFT of the fine scale equals the W1 X W1^T product it stands for
    W1, C1 = tabs['scr_W1'], tabs['scr_C1']
    z1 = rng.standard_normal((64, 64)) + 1j * rng.standard_normal((64, 64))
    z2 = np.zeros((48, 48))
    s = synthesize_screen(tabs, z1, z2, 1.0)
    np.testing.assert_allclose(s, (W1 @ (C1 * z1) @ W1.T).real.ravel(), rtol=0, atol=1e-12 * np.abs(s).max())


@pytest.mark.parametrize('seed', [0, 2 ** 63 - 1])
def test_streams_are_distinct_per_env_draw_and_domain(seed):
    """No two streams of the model share a block: envs, draws, and the extrusion / synthesis domains."""
    blocks = set()
    for env in (0, 1, 1 << 32):
        for draw in (0, 1):
            c, k = extrusion_blocks(seed, env, draw, 240)
            blocks.update(map(bytes, philox4x32_10(c, k)))
    c, k = synthesis_blocks(seed, 0, 0, 16, 4)
    blocks.update(map(bytes, philox4x32_10(c, k)))
    assert len(blocks) == 3 * 2 * 60 + (256 + 16) // 2
