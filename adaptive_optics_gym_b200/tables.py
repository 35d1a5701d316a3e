"""Set-up tables for the B200 ``AO-v0`` step path (host side, NumPy FP64).

Everything the reference computes once at construction time inside hcipy
(``AOEnv.__init__`` -> ``pupil_simulation`` / ``incoming_wavefront`` / ``DM_function`` /
``atmospheric_turbulence`` / ``fiber_coupling``, reference ``gym_AO/envs/AO_env.py:17-71,
293-393``) is table data for the CUDA step kernels.  This module builds those tables
directly in the layouts the kernels read; it shares no code with ``oracle/``.

Any table can be overridden through ``AOEnv(tables={...})`` -- e.g. tables exported from a
real hcipy==0.5.1 install -- which is what keeps the step path faithful even where a
set-up routine (mode ordering, AR matrices, LP solver) is restated rather than run.
"""
from __future__ import annotations

import heapq
from dataclasses import dataclass, field

import numpy as np
from scipy import optimize, special


@dataclass
class AOConfig:
    """Physical constants of ``AOEnv.parameters_init`` (reference AO_env.py:211-247)."""
    atm_type: str = 'quasi_static'
    velocity: float = 0.0
    fried_parameter: float = 0.15
    act_type: str = 'num_actuators'
    num_modes: int = 64
    obs_dim: int = 2
    rew_type: str = 'strehl_ratio'
    max_steps: int = 20
    telescope_diameter: float = 0.5
    num_pupil_pixels: int = 240
    wavelength_wfs: float = 1.5e-6
    wavelength_sci: float = 2.2e-6
    delta_t: float = 1e-3
    outer_scale: float = 10.0
    D_pupil_fiber: float = 0.5
    num_focal_pixels_fiber: int = 128
    multimode_fiber_core_radius: float = 25e-6
    singlemode_fiber_core_radius: float = 4.5e-6
    fiber_NA: float = 0.14
    fiber_length: float = 10.0
    f_number: float = 50.0
    num_lenslets: int = 12
    sh_diameter: float = 5e-3
    stellar_magnitude: float = -5.0
    ssim_ref_peak: float = 2.8          # AO_env.py:492
    stencil_length: int = 2


@dataclass
class AOTables:
    cfg: AOConfig
    scalars: dict = field(default_factory=dict)
    arrays: dict = field(default_factory=dict)

    def __getitem__(self, k):
        return self.arrays[k] if k in self.arrays else self.scalars[k]


# ---------------------------------------------------------------- grids
def pupil_coords(n, diameter):
    """Cell-centred symmetric samples (hcipy make_pupil_grid; AO_env.py:300)."""
    d = diameter / n
    return (np.arange(n) + 0.5) * d - diameter / 2, d


def _mft_pair(out_x, out_y, in_x, in_y, scale, weight):
    """Separable DFT matrices of F[v,u] = sum E[y,x] exp(-i s (u x + v y)) w."""
    m1 = np.exp(-1j * scale * np.outer(out_y, in_y)) * weight      # [Nv, Ny]
    m2 = np.exp(-1j * scale * np.outer(in_x, out_x))               # [Nx, Nu]
    return m1, m2


# ---------------------------------------------------------------- DM modes
def zernike_noll(j):
    """Noll index -> (n, m), sign convention of hcipy (odd j -> sine / negative m)."""
    n = int(np.sqrt(2 * j - 1) + 0.5) - 1
    if n % 2:
        m = 2 * int((2 * (j + 1) - n * (n + 1)) // 4) - 1
    else:
        m = 2 * int((2 * j + 1 - n * (n + 1)) // 4)
    return n, (-m if j % 2 else m)


def zernike_modes(k, diameter, x, y):
    """Noll 1..k on the flat grid (AO_env.py:346), radial part through Jacobi
    polynomials: R_n^m(r) = (-1)^((n-m)/2) r^m P^{(m,0)}_{(n-m)/2}(1 - 2 r^2)."""
    rho = 2 * np.hypot(x, y) / diameter
    th = np.arctan2(y, x)
    inside = rho <= 1
    rc = np.where(inside, rho, 0.0)
    out = np.empty((k, x.size))
    for j in range(1, k + 1):
        n, m = zernike_noll(j)
        am = abs(m)
        s = (n - am) // 2
        rad = (-1) ** s * rc ** am * special.eval_jacobi(s, am, 0, 1 - 2 * rc ** 2)
        az = 1.0 if m == 0 else (np.sqrt(2) * np.cos(am * th) if m > 0 else np.sqrt(2) * np.sin(am * th))
        out[j - 1] = np.sqrt(n + 1) * rad * az * inside
    return out


def disk_harmonic_orders(k):
    """Energy-ordered (n, m) list of the Neumann disk harmonics as hcipy 0.5.1 enumerates
    them: a frontier seeded at (1, 0); the lowest-energy entry is popped (first-inserted wins
    ties), emits the sine copy then the cosine copy when m != 0, and pushes (n, m+1) and
    (n+1, m) unless that order is CURRENTLY on the frontier.  Because membership is tested
    against the live frontier only, an order popped early is pushed again by its second
    parent -- e.g. (2, +-1) appears twice within the first 20 Neumann modes.  That is the
    restated hcipy behaviour [VERIFY against a real install]; ``tables={'dm_modes': ...}``
    overrides it."""
    def energy(n, m):
        return float(special.jnp_zeros(m, n)[-1] ** 2)
    heap = [(energy(1, 0), 0, (1, 0))]
    frontier = {(1, 0)}
    tick = 1
    out = []
    while len(out) < k:
        _, _, (n, m) = heapq.heappop(heap)
        frontier.discard((n, m))
        if m:
            out.append((n, -m))
        out.append((n, m))
        for nm in ((n, m + 1), (n + 1, m)):
            if nm not in frontier:
                frontier.add(nm)
                heapq.heappush(heap, (energy(*nm), tick, nm))
                tick += 1
    return out[:k]


def disk_harmonic_modes(k, diameter, x, y):
    """Neumann disk harmonics J_m(l_mn 2r/D) {cos, sin}(m theta) inside the aperture
    (AO_env.py:352).  Overall scale is irrelevant: the caller divides by peak-to-valley."""
    rho = 2 * np.hypot(x, y) / diameter
    th = np.arctan2(y, x)
    inside = (x * x + y * y) <= (diameter / 2) ** 2
    out = np.empty((k, x.size))
    for i, (n, m) in enumerate(disk_harmonic_orders(k)):
        am = abs(m)
        lam = special.jnp_zeros(am, n)[-1]
        z = special.jv(am, lam * rho) * (np.sin(am * th) if m < 0 else np.cos(am * th))
        out[i] = z * inside
    return out


# ---------------------------------------------------------------- LP fibre modes
def lp_modes(xf, weight, core_radius, NA, wavelength):
    """Guided LP modes of a step-index fibre sampled on the separable focal grid ``xf``
    (hcipy StepIndexFiber / make_LP_modes; AO_env.py:393).  Characteristic equation in
    the standard form u J_{m-1}(u)/J_m(u) + w K_{m-1}(w)/K_m(w) = 0, bracketed between
    consecutive zeros of J_m.  Returns modes [J, Nf*Nf] (unit power on the grid), beta [J]."""
    V = 2 * np.pi / wavelength * core_radius * NA
    k0 = 2 * np.pi / wavelength
    X, Y = np.meshgrid(xf, xf)
    R = (np.hypot(X, Y) / core_radius).ravel()
    TH = np.arctan2(Y, X).ravel()

    def g(u, m):
        w = np.sqrt(V * V - u * u)
        return u * special.jv(m - 1, u) * special.kn(m, w) + w * special.kn(m - 1, w) * special.jv(m, u)

    modes, betas = [], []
    m = 0
    while True:
        # brackets: (previous zero of J_m, next zero of J_m) clipped to (0, V)
        zeros = [z for z in special.jn_zeros(m, 64) if z < V]
        edges = [1e-9] + zeros + [V - 1e-9]
        roots = []
        for a, b in zip(edges[:-1], edges[1:]):
            a2, b2 = a + 1e-9, b - 1e-9
            if a2 < b2 and g(a2, m) * g(b2, m) < 0:
                roots.append(optimize.brentq(g, a2, b2, args=(m,), xtol=1e-15, rtol=8.9e-16))
        if not roots:
            break
        for u in roots:
            w = np.sqrt(V * V - u * u)
            core = R < 1
            rad = np.where(core, special.jv(m, u * np.minimum(R, 1.0)),
                           special.jv(m, u) / special.kn(m, w) * special.kn(m, w * np.maximum(R, 1.0)))
            for az in ([np.cos(m * TH), np.sin(-m * TH)] if m else [np.ones_like(TH)]):
                p = rad * az
                modes.append(p / np.sqrt(np.sum(p * p) * weight))
                betas.append(np.sqrt(k0 * k0 - (u / core_radius) ** 2))
        m += 1
    return np.array(modes), np.array(betas)


# ---------------------------------------------------------------- atmosphere
def cn2_from_fried(r0, wavelength):
    return r0 ** (-5.0 / 3) / (0.423 * (2 * np.pi / wavelength) ** 2)


# Smallest Fried parameter accepted per env.  The tensor / fused paths hold the phase S / lambda_wfs as int32 fixed point
# that saturates at +-512 half-turns (1608 rad).  A screen scales as r0^(-5/6); at r0 = 0.20 m the largest |S| / lambda_wfs
# of 400 synthesised 240 x 240 screens is 33 rad (piston included: the 10 m outer scale gives each screen an offset of
# ~11 rad RMS).  Budgeting 100 rad at 0.20 m (3x that, and 9 sigma of the offset), the clamp is reached at
# r0 = 0.20 (100 / 1608)^(6/5) = 7.1 mm; the floor rounds that up to 1 cm, where the observed maximum (400 rad) is 4x
# below the clamp.
FRIED_MIN = 0.01


def sqrt_cn2_from_fried(r0s, wavelength):
    """sqrt(Cn^2) of each r0, converted one Python float at a time: entry i equals, bit for bit, the value a handle built
    with the scalar r0s[i] uses (a vectorised power may round the last bit differently)."""
    return np.array([float(np.sqrt(cn2_from_fried(float(r), wavelength))) for r in r0s], dtype=np.float64)


def von_karman_covariance(r, r0, L0):
    r = r + 1e-10
    q = 2 * np.pi * r / L0
    c = (special.gamma(11 / 6) / (2 ** (5 / 6) * np.pi ** (8 / 3))) * (24 / 5 * special.gamma(6 / 5)) ** (5 / 6)
    return (L0 / r0) ** (5 / 3) * c * q ** (5 / 6) * special.kv(5 / 6, q)


def ar_extrusion_tables(n, delta, L0, rng, stencil_length=2, extra_columns=None):
    """Horizontal autoregressive extrusion operator of hcipy's InfiniteAtmosphericLayer
    (AO_env.py:370): stencil = first ``stencil_length`` columns plus one pixel per row at
    column g + stencil_length - 1 (g ~ Geometric(1/2), drawn once), sorted by flat index;
    new column x = -1:  col = A z + sqrt(Cn2) B xi.  Covariances at Cn2 = 1, lambda = 1 m.

    Returns (stencil_flat_idx [n_s] int32, A [n, n_s], B [n, n])."""
    sl = stencil_length
    extra = (rng.geometric(0.5, n) + sl - 1) % n if extra_columns is None else np.asarray(extra_columns)
    cols = np.concatenate([np.tile(np.arange(sl), n), extra])
    rows = np.concatenate([np.repeat(np.arange(n), sl), np.arange(n)])
    flat = np.unique(rows * n + cols)
    sy, sx = flat // n, flat % n
    px = np.concatenate([sx.astype(float), np.full(n, -1.0)]) * delta
    py = np.concatenate([sy.astype(float), np.arange(n, dtype=float)]) * delta
    r0 = (0.423 * (2 * np.pi) ** 2) ** (-3.0 / 5)
    cov = von_karman_covariance(np.hypot(px[:, None] - px[None, :], py[:, None] - py[None, :]), r0, L0)
    ns = flat.size
    U, S, Vt = np.linalg.svd(cov[:ns, :ns], full_matrices=False)
    zz_inv = (Vt.T * (S / (S * S + (1e-10 * S.max()) ** 2))) @ U.T
    A = cov[ns:, :ns] @ zz_inv
    Ub, Sb, _ = np.linalg.svd(cov[ns:, ns:] - A @ cov[:ns, ns:])
    return flat.astype(np.int32), A, Ub * np.sqrt(Sb)


def screen_synthesis_tables(n, delta, L0, oversampling=16):
    """Spectral amplitudes for von-Karman screen synthesis at Cn2 = 1, lambda = 1 m
    (hcipy FiniteAtmosphericLayer(oversampling=16) behind InfiniteAtmosphericLayer's
    initial screen / ``reset()``; AO_env.py:77,370).  Two scales: the n x n DFT grid without
    its central 3x3 bins, and a 3*os x 3*os grid ``oversampling`` times finer covering them.
    screen = Re[W1 (C1 . xi1) W1^T] + Re[W2 (C2 . xi2) W2^T], xi complex standard normal."""
    r0 = (0.423 * (2 * np.pi) ** 2) ** (-3.0 / 5)
    x, _ = pupil_coords(n, n * delta)

    def amp(fx, fy, df):
        return np.sqrt(0.0229 * r0 ** (-5 / 3) * (fx ** 2 + fy ** 2 + L0 ** -2) ** (-11 / 6)) * df

    df1 = 1.0 / (n * delta)
    k1 = np.fft.fftfreq(n, d=1.0 / n)
    KX, KY = np.meshgrid(k1, k1)
    C1 = amp(KX * df1, KY * df1, df1)
    C1[(np.abs(KX) <= 1) & (np.abs(KY) <= 1)] = 0
    W1 = np.exp(2j * np.pi * np.outer(x, k1 * df1))
    n2 = 3 * oversampling
    df2 = df1 / oversampling
    f2 = (np.arange(n2) + 0.5 - n2 / 2) * df2
    FX, FY = np.meshgrid(f2, f2)
    C2 = amp(FX, FY, df2)
    W2 = np.exp(2j * np.pi * np.outer(x, f2))
    return dict(scr_C1=C1, scr_W1=W1, scr_C2=C2, scr_W2=W2)


def synthesize_screens(tabs, num, cn2, rng):
    """Host-side screen synthesis from ``screen_synthesis_tables`` (construction time and
    CPU tests; the per-episode ``semi_dynamic`` regeneration runs on the GPU)."""
    C1, C2 = tabs['scr_C1'], tabs['scr_C2']
    out = np.empty((num, C1.size))
    for i in range(num):
        z1 = rng.standard_normal(C1.shape) + 1j * rng.standard_normal(C1.shape)
        z2 = rng.standard_normal(C2.shape) + 1j * rng.standard_normal(C2.shape)
        out[i] = synthesize_screen(tabs, z1, z2, np.sqrt(cn2))
    return out


def synthesize_screen(tabs, z1, z2, sqrt_cn2):
    """One screen [y][x] (flattened) of ``synthesize_screens`` from given complex normals: z1 [n][n] and z2 [n2][n2],
    indexed [ky][kx] like the tables."""
    C1, W1, C2, W2 = tabs['scr_C1'], tabs['scr_W1'], tabs['scr_C2'], tabs['scr_W2']
    n = C1.shape[0]
    # W1 is a (shifted) DFT: use the FFT for the fine grid
    sh = W1[0, :]                                      # exp(2 pi i f_k x_0)
    s = (np.fft.ifft2(C1 * z1 * sh[None, :] * sh[:, None]) * n * n).real
    s += (W2 @ (C2 * z2) @ W2.T).real
    return s.ravel() * sqrt_cn2


# ---------------------------------------------------------------- everything
def build_tables(cfg: AOConfig, rng=None, overrides=None) -> AOTables:
    rng = np.random.default_rng(0) if rng is None else rng
    t = AOTables(cfg)
    A, S = t.arrays, t.scalars
    Np, D = cfg.num_pupil_pixels, cfg.telescope_diameter
    xp, dp = pupil_coords(Np, D)
    X = np.tile(xp, Np)
    Y = np.repeat(xp, Np)
    ap = ((X * X + Y * Y) <= (D / 2) ** 2).astype(np.float64)
    n_ap = float(ap.sum())
    w_p = dp * dp
    A['aperture'] = ap
    S.update(num_aperture_pixels=n_ap, pupil_delta=dp, pupil_weight=w_p)

    # incoming wavefronts (AO_env.py:319-334): E0 = A sqrt(P_tot / (N_ap w))
    flux = 3.9e10 * 10 ** (-cfg.stellar_magnitude / 2.5)
    S['amp_fiber'] = np.sqrt(1.0 / (n_ap * w_p))
    S['amp_flux'] = np.sqrt(flux / (n_ap * w_p))
    S['total_flux'] = flux

    # DM (AO_env.py:339-358): modes / ptp(mode)
    modes = (zernike_modes if cfg.act_type == 'zernike' else disk_harmonic_modes)(cfg.num_modes, D, X, Y)
    modes = modes / np.ptp(modes, axis=1, keepdims=True)
    A['dm_modes'] = modes                                             # [K, P]
    mean = modes.mean(axis=1)
    A['dm_gram'] = modes @ modes.T / modes.shape[1] - np.outer(mean, mean)   # var(M a) = a^T G a

    # fibre arm (AO_env.py:373-393)
    Df = 2.1 * cfg.multimode_fiber_core_radius
    f_fib = cfg.D_pupil_fiber / (2 * cfg.fiber_NA)
    xf, df = pupil_coords(cfg.num_focal_pixels_fiber, Df)
    xo, do = pupil_coords(cfg.obs_dim, Df)
    sc = 2 * np.pi / (f_fib * cfg.wavelength_wfs)
    A['mft_fib_1'], A['mft_fib_2'] = _mft_pair(xf, xf, xp, xp, sc, w_p)
    A['mft_obs_1'], A['mft_obs_2'] = _mft_pair(xo, xo, xp, xp, sc, w_p)
    S['mft_fib_norm'] = 1.0 / (1j * f_fib * cfg.wavelength_wfs)
    S.update(fiber_focal_weight=df * df, obs_weight=do * do, fiber_focal_length=f_fib)
    lp, beta = lp_modes(xf, df * df, cfg.singlemode_fiber_core_radius, cfg.fiber_NA, cfg.wavelength_wfs)
    A['lp_modes_w'] = lp * (df * df)                                  # [J, Nf^2]  mode * weight
    A['lp_phase'] = np.exp(1j * beta * cfg.fiber_length)              # [J]
    A['lp_gram'] = (lp @ lp.T) * (df * df)                            # [J, J]
    A['lp_beta'] = beta

    # science arm / Strehl (AO_env.py:313-321, 479-483): the reference reads ONE focal pixel,
    # argmax of the unaberrated PSF.  With the focal grid sampled at the origin that pixel is
    # (u, v) = (0, 0) and P[idx] = |amp w_p sum_ap exp(i phi)|^2 D_f^2 / (lambda f)^2.
    res = cfg.wavelength_sci / D
    nfoc = int(2 * 30 * 4)
    dfoc = res / 4
    xs = dfoc * (np.arange(nfoc) - nfoc / 2 + (nfoc % 2) * 0.5)
    i0 = int(np.argmin(np.abs(xs)))
    if abs(xs[i0]) > 1e-12 * dfoc:
        raise ValueError('science focal grid has no sample at the origin')
    # Both powers carry the same amp^2 w_p^2 D_f^2 / lambda^2 factor and P_tot ratio, so
    # strehl[%] = 100 |sum_ap exp(i phi)|^2 / N_ap^2.
    S['strehl_scale'] = 100.0 / (n_ap * n_ap)
    S['sci_focal_index'] = i0 * nfoc + i0
    A['sci_focal_coords'] = xs

    # atmosphere (AO_env.py:361-370)
    cn2 = cn2_from_fried(cfg.fried_parameter, cfg.wavelength_sci)
    S['cn2'] = cn2
    if cfg.atm_type == 'dynamic':
        A['ar_stencil'], A['ar_A'], A['ar_B'] = ar_extrusion_tables(Np, dp, cfg.outer_scale, rng, cfg.stencil_length)
    A.update(screen_synthesis_tables(Np, dp, cfg.outer_scale))

    if overrides:
        for k, v in overrides.items():
            (A if isinstance(v, np.ndarray) else S)[k] = v
    return t


# ---------------------------------------------------------------- Shack-Hartmann (SH_operation=True)
def build_sh_tables(cfg: AOConfig, T: AOTables) -> dict:
    """Tables of the Shack-Hartmann integrator (reference ``shack_hartmann_init``, AO_env.py:396-465, and
    ``SH_step``, :254-290).

    hcipy chain restated: ``Magnifier(m)`` (grid x m, field / m), ``SquareShackHartmannWavefrontSensorOptics``
    (lenslet centres ``arange(-D_sh, D_sh, D_sh/12)``, nearest-lenslet phase ``-k d^2 / (2 f)``, ``f = 50 pitch``),
    ``FresnelPropagator`` over ``f`` -- an angular-spectrum filter with a 2x zero-padded FFT whose transfer
    function factorises in x and y, so pad -> FFT -> filter -> IFFT -> crop is the separable linear map
    ``E_out = C E C^T`` with one precomputed ``C [Np, Np]`` -- ``NoiselessDetector`` (image = power x dt,
    carried on the science focal grid, :412) and the flux-weighted centroid estimator.  Calibration (sub-aperture
    selection at half the peak flux, reference slopes, push-pull interaction matrix at 0.01 lambda, Tikhonov
    inverse rcond 1e-3) runs here on the host once, through the same ``C``.
    """
    Np, D = cfg.num_pupil_pixels, cfg.telescope_diameter
    lam = cfg.wavelength_wfs
    k = 2 * np.pi / lam
    mag = cfg.sh_diameter / D
    xp, dp = pupil_coords(Np, D)
    xs, ds = xp * mag, dp * mag
    pitch = cfg.sh_diameter / cfg.num_lenslets
    cen = np.arange(-cfg.sh_diameter, cfg.sh_diameter, pitch)
    nl = cen.size
    near = np.argmin(np.abs(xs[:, None] - cen[None, :]), axis=1)              # lenslet of each pixel, per axis
    lens_of_pixel = (near[:, None] * nl + near[None, :]).ravel()             # [y][x] flat
    f = cfg.f_number * pitch
    d2 = ((xs - cen[near]) ** 2)
    mla_phase = (-(d2[:, None] + d2[None, :]) / (2 * f) * k).ravel()

    q = 2 * np.pi * np.fft.fftfreq(2 * Np, d=ds)
    h1 = np.exp(-0.5j * (f / k) * q * q)
    pad = np.zeros((2 * Np, Np), dtype=np.complex128)
    pad[Np // 2:Np // 2 + Np, :] = np.eye(Np)
    C = np.fft.ifft(h1[:, None] * np.fft.fft(pad, axis=0), axis=0)[Np // 2:Np // 2 + Np, :]

    xs_det = T['sci_focal_coords']                                            # the detector grid the reference passes
    if xs_det.size != Np:
        raise ValueError('SH_operation needs num_pupil_pixels == 240 (the reference reads the camera on the '
                         '240 x 240 science focal grid, AO_env.py:412)')
    gx, gy = np.tile(xs_det, Np), np.repeat(xs_det, Np)
    ap = T['aperture']

    def image(E_pupil, dt):
        e = (E_pupil / mag * np.exp(1j * mla_phase)).reshape(Np, Np)
        out = C @ e @ C.T
        return (np.abs(out) ** 2).ravel() * (ds * ds) * dt

    def sums(img, lenslets):
        fl = np.bincount(lens_of_pixel, weights=img, minlength=nl * nl)[lenslets]
        sx = np.bincount(lens_of_pixel, weights=img * gx, minlength=nl * nl)[lenslets]
        sy = np.bincount(lens_of_pixel, weights=img * gy, minlength=nl * nl)[lenslets]
        return fl, sx, sy

    # reference image of the bare aperture (unit amplitude, dt = 1; AO_env.py:413-415)
    img_ref = image(ap.astype(np.complex128), 1.0)
    present = np.unique(lens_of_pixel)
    flux, _, _ = sums(img_ref, present)
    selected = present[flux > 0.5 * flux.max()]
    centres = np.array((np.tile(cen, nl)[selected], np.repeat(cen, nl)[selected]))

    def slopes(img):
        fl, sx, sy = sums(img, selected)
        return np.array((sx / fl, sy / fl)) - centres

    slopes_ref = slopes(img_ref)
    modes = T['dm_modes']                                                     # [K, P]
    probe = 0.01 * lam
    E_cal = T['amp_fiber'] * ap
    resp = []
    for i in range(cfg.num_modes):
        acc = 0
        for amp in (-probe, probe):
            acc = acc + amp * slopes(image(E_cal * np.exp(2j * k * amp * modes[i]), 1.0)) / probe ** 2
        resp.append(acc.ravel())
    resp = np.stack(resp, axis=1)                                             # [2 Nsub, K]
    U, S, Vt = np.linalg.svd(resp, full_matrices=False)
    recon = (Vt.T * (S / (S * S + (1e-3 * S.max()) ** 2))) @ U.T              # [K, 2 Nsub]

    # per selected lenslet: CSR list of its pixels (deterministic warp reductions on the device)
    order = np.argsort(lens_of_pixel, kind='stable')
    slot_of_lens = np.full(nl * nl, -1)
    slot_of_lens[selected] = np.arange(selected.size)
    keep = order[slot_of_lens[lens_of_pixel[order]] >= 0]
    slots = slot_of_lens[lens_of_pixel[keep]]
    offsets = np.concatenate(([0], np.cumsum(np.bincount(slots, minlength=selected.size)))).astype(np.int32)
    act0 = np.zeros(cfg.num_modes)
    act0[-1] = probe          # the calibration loop leaves its last probe on the SH mirror (AO_env.py:446-447)
    return dict(
        sh_mla_phase=mla_phase, sh_fresnel=C, sh_pix_offsets=offsets, sh_pix_index=keep.astype(np.int32),
        sh_pix_x=gx[keep], sh_pix_y=gy[keep], sh_offset=(centres + slopes_ref), sh_recon=recon, sh_act0=act0,
        sh_amplitude=float(T['amp_flux'] / mag), sh_weight_dt=float(ds * ds * cfg.delta_t),
        sh_num_sub=int(selected.size), sh_selected=selected, sh_slopes_ref=slopes_ref, sh_response=resp,
    )
