"""``AOEnv`` / ``AOVecEnv`` -- the ``AO-v0`` boundary of the reference on B200 CUDA kernels.

``AOEnv`` mirrors ``gym_AO.envs.AO_env.AOEnv`` of the reference (constructor kwargs
``AO_env.py:17-29``; ``reset`` ``:74-103``; ``step`` ``:106-153``; ``SH_step`` ``:254-290``;
``render`` ``:156-194``): same names, argument meaning, return types and error behaviour, so
``main.py`` / ``algorithm.py`` / ``eval_policy.py`` run unchanged against it.  ``AOVecEnv`` is the
vectorised N-environment variant (not in the reference): the same kwargs plus ``num_envs``, torch
CUDA tensors in and out, all environments in lock-step.

All arithmetic of reset/step runs in ``libaogym.so`` (hand-written sm_100a CUDA behind the C-ABI
of ``include/aogym.h``); this file only builds the set-up tables and marshals buffers.  There is
no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._gym_compat import Env, spaces
from .tables import FRIED_MIN, AOConfig, build_sh_tables, build_tables, sqrt_cn2_from_fried, synthesize_screens


def _coerce_velocity(atm_type, velocity_value):
    """Reference AO_env.py:200-208 (including its two prints)."""
    if (atm_type == 'quasi_static' or atm_type == 'semi_dynamic') and velocity_value != 0:
        print('In ' + atm_type + ' atmospheric condition, the velocity value should be zero.')
        print('therefore velocity value is changed to zero')
        velocity_value = 0
    elif atm_type == 'dynamic' and velocity_value == 0:
        print('In ' + atm_type + ' atmospheric condition, the velocity value cannot be zero.')
        print('therefore velocity value is changed to 1 m/s')
        velocity_value = 1
    return velocity_value


def fried_values(r0, num_envs):
    """A Fried parameter given per env -> (float64 [num_envs], was a scalar).  ``r0``: a scalar (broadcast), or a
    sequence, NumPy array or tensor (a CUDA tensor is copied to the host) of ``num_envs`` values, each finite and at
    least ``FRIED_MIN`` m (below it the fixed-point phase of the tensor / fused paths could saturate)."""
    if hasattr(r0, 'detach'):
        r0 = r0.detach().cpu().numpy()
    a = np.asarray(r0, dtype=np.float64)
    scalar = a.ndim == 0
    if scalar:
        a = np.full(num_envs, float(a))
    if a.shape != (num_envs,):
        raise ValueError(f'atm_fried must be a scalar or {num_envs} values (one per env), got shape {a.shape}')
    if not np.all(np.isfinite(a)) or np.any(a <= 0):
        raise ValueError('atm_fried values must be finite and positive')
    if np.any(a < FRIED_MIN):
        raise ValueError(f'atm_fried values must be >= {FRIED_MIN} m (the fixed-point phase saturates below it)')
    return a, scalar


class _AOCore:
    """Shared construction: config -> tables -> device handle -> initial screens."""

    def _setup(self, *, atm_type, atm_vel, atm_fried, act_type, act_dim, obs_dim, rew_type, rew_threshold,
               timesteps_per_episode, flat_mirror_start_per_episode, SH_operation, num_envs, device, seed,
               precision, tables, initial_screens, num_pupil_pixels, num_focal_pixels_fiber, env_id_base):
        if atm_type not in _lib.ATM:
            raise ValueError(f'atm_type must be one of {list(_lib.ATM)}')
        # arithmetic of the step path: the kwarg, else $AOG_PRECISION (so that the reference's unchanged
        # ``gym.make('AO-v0', ...)`` call can select the fast path), else the exact FP64 kernels
        if precision is None:
            precision = os.environ.get('AOG_PRECISION', 'f64')
        if precision not in _lib.PRECISION:
            raise ValueError(f'precision must be one of {list(_lib.PRECISION)}')
        self.precision = precision
        self.atm_type = atm_type
        self.rew_type = rew_type
        self.act_type = act_type
        self.flat_mirror_start_per_episode = flat_mirror_start_per_episode
        self.rew_threshold = rew_threshold
        self.SH_operation = SH_operation
        self.num_envs = int(num_envs)
        # a scalar keeps the handle-wide value of cfg.sqrt_cn2; a sequence is validated here, before any device call
        fried = None if np.ndim(atm_fried) == 0 else fried_values(atm_fried, self.num_envs)[0]
        velocity = _coerce_velocity(atm_type, atm_vel)
        cfg = AOConfig(atm_type=atm_type, velocity=float(velocity),
                       fried_parameter=float(atm_fried) if fried is None else float(fried[0]),
                       act_type=act_type, num_modes=int(act_dim), obs_dim=int(obs_dim), rew_type=rew_type,
                       max_steps=int(timesteps_per_episode), num_pupil_pixels=int(num_pupil_pixels),
                       num_focal_pixels_fiber=int(num_focal_pixels_fiber))
        self.config = cfg
        # reference attribute names (AO_env.py:249-251 assigns every parameter onto self)
        for k in ('telescope_diameter', 'num_pupil_pixels', 'wavelength_wfs', 'wavelength_sci', 'num_modes',
                  'delta_t', 'max_steps', 'velocity', 'fried_parameter', 'outer_scale',
                  'singlemode_fiber_core_radius', 'multimode_fiber_core_radius'):
            setattr(self, k, getattr(cfg, k))
        if fried is not None:
            self.fried_parameter = fried.copy()
        self.num_focal_pixels_fiber = cfg.num_focal_pixels_fiber
        self.num_focal_pixels_fiber_subsample = cfg.obs_dim
        # The reference draws its screens and noise from NumPy's unseeded global generator (every construction is a
        # new atmosphere), so seed=None takes fresh entropy; only an explicit seed is deterministic.  The seed in
        # use is kept on the env (``seed_used``) so a run can be reproduced afterwards.
        self._seed = (int(np.random.SeedSequence().entropy) & (2 ** 63 - 1)) if seed is None else int(seed)
        self.seed_used = self._seed
        rng = np.random.default_rng(self._seed)
        self.tables = build_tables(cfg, rng=rng, overrides=tables)
        t = self.tables

        # skimage raises ValueError from step() when obs_dim^2 < 7 (AO_env.py:495); keep that
        # behaviour at the boundary and give the device a configuration it accepts.
        self._ssim_too_small = rew_type == 'smf_ssim' and cfg.obs_dim ** 2 < 7
        if rew_type not in _lib.REW:
            raise ValueError(f'rew_type must be one of {list(_lib.REW)}')

        c = _lib.AogConfig()
        c.abi_version = _lib.ABI_VERSION
        c.device = int(device)
        c.num_envs = self.num_envs
        c.num_pupil_pixels = cfg.num_pupil_pixels
        c.num_focal_pixels = cfg.num_focal_pixels_fiber
        c.obs_dim = cfg.obs_dim
        c.num_modes = cfg.num_modes
        c.num_lp_modes = int(t['lp_phase'].size)
        c.num_stencil = int(t['ar_stencil'].size) if 'ar_stencil' in t.arrays else 0
        c.num_screen_fine = int(t['scr_C2'].shape[0])
        c.atm_type = _lib.ATM[atm_type]
        c.rew_type = _lib.REW['strehl_ratio'] if self._ssim_too_small else _lib.REW[rew_type]
        c.sh_operation = int(bool(SH_operation))
        c.flat_mirror_start = int(bool(flat_mirror_start_per_episode))
        c.max_steps = cfg.max_steps
        c.has_rew_threshold = int(rew_threshold is not None)
        c.rew_threshold = float(rew_threshold) if rew_threshold is not None else 0.0
        c.precision = _lib.PRECISION[precision]
        c.env_id_base = int(env_id_base)
        c.wavelength_wfs = cfg.wavelength_wfs
        c.wavelength_sci = cfg.wavelength_sci
        c.delta_t = cfg.delta_t
        c.velocity = cfg.velocity
        c.pupil_delta = t['pupil_delta']
        c.amp_fiber = t['amp_fiber']
        c.sqrt_cn2 = float(np.sqrt(t['cn2']))
        c.strehl_scale = t['strehl_scale']
        c.obs_weight = t['obs_weight']
        c.ssim_ref_peak = cfg.ssim_ref_peak
        c.mft_norm_re = float(np.real(t['mft_fib_norm']))
        c.mft_norm_im = float(np.imag(t['mft_fib_norm']))
        c.seed = self._seed
        self._h = _lib.Handle(c)
        for name in _lib.TABLE_IDS:
            if name in t.arrays and not name.startswith('sh_'):
                self._h.set_table(name, t.arrays[name])
        # Shack-Hartmann integrator (AO_env.py:396-465): calibrated on the host once, tables on the device
        self.sh_tables = None
        if SH_operation:
            sh = build_sh_tables(cfg, t)
            if tables:
                sh.update({k: v for k, v in tables.items() if k.startswith('sh_')})
            self.sh_tables = sh
            self._h.sh_configure(sh['sh_num_sub'], sh['sh_pix_index'].size, sh['sh_amplitude'], sh['sh_weight_dt'])
            for name in _lib.TABLE_IDS:
                if name.startswith('sh_'):
                    self._h.set_table(name, sh[name])
        if fried is not None:
            self._h.set_turbulence(sqrt_cn2_from_fried(fried, cfg.wavelength_sci))
        # initial screen(s) (hcipy draws one at construction; AO_env.py:370)
        if initial_screens is not None:
            s = np.asarray(initial_screens)
            s = s.reshape(-1, cfg.num_pupil_pixels ** 2)
            if s.shape[0] == 1 and self.num_envs > 1:
                s = np.repeat(s, self.num_envs, axis=0)
            if s.shape[0] != self.num_envs:
                raise ValueError('initial_screens must hold one screen per env')
            self._h.set_screens(s)
        else:
            self._h.generate_screens()
        self.timestep = 0
        self.episode_no = 0
        self.timestep_render = 0

    # ---- state shared by both front ends
    def _stream(self):
        return 0

    def _set_fried(self, r0, rescale):
        """New per-env Fried parameters for every later screen synthesis and extrusion; ``rescale`` also scales each
        env's current screen by (r0_old / r0_new)^(5/6): the same realisation at the new strength."""
        vals, scalar = fried_values(r0, self.num_envs)
        self._h.set_turbulence(sqrt_cn2_from_fried(vals, self.wavelength_sci), rescale, self._stream())
        self.fried_parameter = float(vals[0]) if scalar else vals

    def _reset_options(self, options):
        """``options={'atm_fried': r0}`` of ``reset``: semi_dynamic draws this reset's screens at the new strength;
        quasi_static and dynamic rescale the screens they keep (for dynamic the AR process is linear in sqrt(Cn^2),
        so later extrusions continue it consistently)."""
        if options and 'atm_fried' in options:
            self._set_fried(options['atm_fried'], rescale=self.atm_type != 'semi_dynamic')

    def _sync_counters(self):
        c = self._h.counters()
        self.timestep, self.timestep_render, self.episode_no = c.timestep, c.timestep_render, c.episode_no

    def get_state(self):
        """Environment state (absent in the reference): screens, DM actuators, the Shack-Hartmann integrator's own
        mirror, counters, and the key + draw counters of every random stream -- a ``set_state`` of this dict on an
        env built with the same kwargs continues bit for bit (device noise included)."""
        c = self._h.counters()
        st = dict(screens=self._h.get_screens(), actuators=self._h.get_actuators(),
                  timestep=c.timestep, timestep_render=c.timestep_render, episode_no=c.episode_no,
                  extrusions=c.extrusions, screen_draws=c.screen_draws, sh_draws=c.sh_draws, seed=self._seed,
                  fried_parameter=np.copy(self.fried_parameter) if np.ndim(self.fried_parameter) else self.fried_parameter)
        if self.SH_operation:
            st['sh_actuators'] = self._h.get_sh_actuators()
        return st

    def set_state(self, state):
        self._h.set_counters(column_origin=0)
        if 'fried_parameter' in state:       # dicts written before per-env strengths existed leave them untouched
            self._set_fried(state['fried_parameter'], rescale=False)
        self._h.set_screens(state['screens'])
        self._h.set_actuators(state['actuators'])
        if 'seed' in state:
            self._reseed(state['seed'])
        if self.SH_operation and 'sh_actuators' in state:
            self._h.set_sh_actuators(state['sh_actuators'])
        self._h.set_counters(timestep=state['timestep'], timestep_render=state['timestep_render'],
                             episode_no=state['episode_no'], extrusions=state['extrusions'], column_origin=0,
                             screen_draws=state.get('screen_draws', 0), sh_draws=state.get('sh_draws', 0))
        self._sync_counters()

    def _reseed(self, seed):
        """Re-key the device's random streams (extrusion noise, screen synthesis, photon noise)."""
        self._seed = int(seed) & (2 ** 63 - 1)
        self.seed_used = self._seed
        self._h.reseed(self._seed)

    def close(self):
        self._h.close()


class AOEnv(_AOCore, Env):
    """Single ``AO-v0`` environment, NumPy in / NumPy out (reference ``AO_env.py:16-503``).

    Extra optional kwargs (defaults = reference constants): ``device``, ``seed``, ``precision``
    ('f64' exact arithmetic, the default | 'fused' one tcgen05 optics kernel per step, ~1e-5 | 'tensor' split-fp16
    tcgen05 matrix Fourier transform, ~1e-5; default taken from ``$AOG_PRECISION``), ``tables`` (override any set-up
    table), ``initial_screen``, ``num_pupil_pixels``, ``num_focal_pixels_fiber``, ``env_id_base`` (the global
    id of this env: the key of its device random streams, so that a single env can replay env i of an ``AOVecEnv``).
    """

    metadata = {'render_modes': ['human']}

    def __init__(self, atm_type='quasi_static', atm_vel=0, atm_fried=0.15, act_type='num_actuators', act_dim=64,
                 obs_dim=2, rew_type='strehl_ratio', rew_threshold=None, timesteps_per_episode=20,
                 flat_mirror_start_per_episode=True, SH_operation=False, *, device=0, seed=None,
                 precision=None, tables=None, initial_screen=None, num_pupil_pixels=240,
                 num_focal_pixels_fiber=128, env_id_base=0):
        super().__init__()
        self._setup(atm_type=atm_type, atm_vel=atm_vel, atm_fried=float(atm_fried), act_type=act_type, act_dim=act_dim,
                    obs_dim=obs_dim, rew_type=rew_type, rew_threshold=rew_threshold,
                    timesteps_per_episode=timesteps_per_episode,
                    flat_mirror_start_per_episode=flat_mirror_start_per_episode, SH_operation=SH_operation,
                    num_envs=1, device=device, seed=seed, precision=precision, tables=tables,
                    initial_screens=initial_screen, num_pupil_pixels=num_pupil_pixels,
                    num_focal_pixels_fiber=num_focal_pixels_fiber, env_id_base=env_id_base)
        # AO_env.py:45-46
        self.observation_space = spaces.Box(low=-1, high=1, shape=(self.num_focal_pixels_fiber_subsample ** 2,),
                                            dtype=np.float16)
        self.action_space = spaces.Box(low=-1, high=1, shape=(self.num_modes,), dtype=np.float16)
        self.last_obs_f64 = None
        self.last_strehl = None
        self.last_ssim = None

    def reset(self, seed=None, options=None):
        """AO_env.py:74-103 -> (float16 obs [obs_dim^2], {}).  The reference ignores ``seed`` (its noise comes from
        NumPy's global generator); here ``seed=s`` re-keys the device's random streams first, so everything drawn from
        this reset on (a ``semi_dynamic`` screen, extrusion noise, photon noise) is reproducible.  The reference
        ignores ``options``; here ``options={'atm_fried': r0}`` (a scalar) sets a new Fried parameter from this reset
        on (see ``AOVecEnv.reset``)."""
        if seed is not None:
            self._reseed(seed)
        self._reset_options(options)
        h = self._h.reset_host()
        self._sync_counters()
        self.last_obs_f64 = h['obs_f64'][0].copy()
        return h['obs_f16'][0].copy(), {}

    def step(self, action, extrusion_noise=None):
        """AO_env.py:106-153 -> (float16 obs, reward, done, False, {"power": float})."""
        if self._ssim_too_small:
            raise ValueError('win_size exceeds image extent. Either ensure that your images are at least 7x7; '
                             'or pass win_size explicitly in the function call, with an odd value less than or '
                             'equal to the smaller side of your images.')
        a = np.asarray(action)
        if a.dtype != np.float32:
            a = a.astype(np.float64)
        if extrusion_noise is None and a.size == self.num_modes:
            h, done = self._h.step_host_fast(np.ascontiguousarray(a))
        else:
            h, done = self._h.step_host(a.reshape(1, -1), extrusion_noise)
        self.timestep += 1                       # AO_env.py:123-124, 149 (the handle keeps the same counters)
        self.timestep_render += 1
        self.episode_no += int(done)
        self.last_obs_f64 = h['obs_f64'][0].copy()
        self.last_strehl = float(h['strehl'][0])
        self.last_ssim = float(h['ssim'][0])
        reward = np.float64(h['reward'][0])
        return h['obs_f16'][0].copy(), reward, done, False, {"power": float(h['power'][0])}

    def SH_step(self, noise='poisson', noisy_image=None):
        """AO_env.py:254-290 -> (action float64 [act_dim], torch.tensor([1])).  The action is the state of the
        integrator's own mirror after ``a <- 0.99 a - 0.3 R slopes``.  Parity-only arguments: ``noise`` =
        'poisson' (device Philox photon noise, the reference's unseeded ``large_poisson``) | 'none' | 'injected'
        (``noisy_image`` [P] = the camera image after photon noise)."""
        if not self.SH_operation:
            raise AttributeError("'AOEnv' object has no attribute 'shwfs'")   # reference: built only with SH_operation
        import torch
        action = self._h.sh_step_host(noise, noisy_image)[0]
        return action, torch.tensor([1])

    def render(self, close=False):
        """AO_env.py:156-194.  Reads the three panels' fields back from the device; draws them when
        matplotlib is importable, and always leaves them in ``self.last_render``."""
        screen = self._h.get_field('screen')
        opd = screen / self.wavelength_wfs * (self.wavelength_wfs / (2 * np.pi)) * 1e6
        self.last_render = dict(phase_screen_opd=opd, focal_power=self._h.get_field('focal_power'),
                                obs_power=self._h.get_field('obs_power'))
        try:
            import matplotlib.pyplot as plt
        except ImportError:
            return
        n, nf, no = self.num_pupil_pixels, self.num_focal_pixels_fiber, self.num_focal_pixels_fiber_subsample
        plt.suptitle('episode %d - timestep %d / %d' % (self.episode_no + 1, self.timestep_render + 1, self.max_steps))
        plt.subplots_adjust(wspace=1, hspace=1)
        plt.subplot(2, 2, 1)
        plt.title(r'Atmospheric phase screen $ [\mu m]$')
        plt.imshow(opd.reshape(n, n), vmin=-6, vmax=6, cmap='RdBu', origin='lower')
        plt.colorbar()
        plt.subplot(2, 2, 3)
        plt.title('Wavefront power on focal plane')
        plt.imshow(self.last_render['focal_power'].reshape(nf, nf), vmin=0, origin='lower')
        plt.colorbar()
        plt.subplot(2, 2, 4)
        plt.title('Wavefront power on photodetector')
        plt.imshow(self.last_render['obs_power'].reshape(no, no), vmin=0, origin='lower')
        plt.colorbar()
        plt.show(block=False)
        plt.pause(0.05)
        plt.clf()


class AOVecEnv(_AOCore):
    """``num_envs`` lock-stepped ``AO-v0`` environments on one B200; torch CUDA tensors in/out.

    ``reset() -> (obs [B, n^2] float16, {})``;
    ``step(actions [B, K]) -> (obs, reward [B] f64, done [B] bool, trunc [B] bool, {"power": [B] f64})``.
    Every env shares ``timesteps_per_episode`` so all terminate on the same step (the caller
    resets after ``done``, as with the single env).  Sharding across GPUs: one instance per rank
    with ``env_id_base = rank * num_envs`` (RNG stream = global env id); no collective on the
    step path.

    ``atm_fried`` is a scalar (every env sees the same turbulence) or one Fried parameter per env (a sequence, NumPy
    array or tensor of ``num_envs`` values, each >= ``tables.FRIED_MIN`` = 1 cm): domain randomisation or evaluation
    across seeing in one batch.  ``fried_parameter`` is then an ``np.ndarray``.  ``reset(options={'atm_fried': r0})``
    changes the values from that episode on.  A sharded run passes each rank its slice ``r0[first:first + count]`` of
    ``sharding.shard_range`` with ``env_id_base = first``, so that env i sees the same r0 and random streams as in one
    handle.

    The tensors returned by ``reset`` / ``step`` / ``SH_step`` (``obs``, ``reward``, ``power``, ``sh_action``, the
    ``done`` masks) are VIEWS OF REUSED OUTPUT BUFFERS: the next call overwrites them in place.  A caller that keeps
    them across calls (a replay buffer, ``next_obs`` bookkeeping) must ``.clone()`` them -- ``rollout.py`` does.
    """

    def __init__(self, num_envs, atm_type='quasi_static', atm_vel=0, atm_fried=0.15, act_type='num_actuators',
                 act_dim=64, obs_dim=2, rew_type='strehl_ratio', rew_threshold=None, timesteps_per_episode=20,
                 flat_mirror_start_per_episode=True, SH_operation=False, *, device=0, seed=None, precision=None,
                 tables=None, initial_screens=None, num_pupil_pixels=240, num_focal_pixels_fiber=128,
                 env_id_base=0):
        import torch
        self._torch = torch
        self.device = torch.device('cuda', int(device))
        self._setup(atm_type=atm_type, atm_vel=atm_vel, atm_fried=atm_fried, act_type=act_type, act_dim=act_dim,
                    obs_dim=obs_dim, rew_type=rew_type, rew_threshold=rew_threshold,
                    timesteps_per_episode=timesteps_per_episode,
                    flat_mirror_start_per_episode=flat_mirror_start_per_episode, SH_operation=SH_operation,
                    num_envs=num_envs, device=device, seed=seed, precision=precision, tables=tables,
                    initial_screens=initial_screens, num_pupil_pixels=num_pupil_pixels,
                    num_focal_pixels_fiber=num_focal_pixels_fiber, env_id_base=env_id_base)
        B, n2 = self.num_envs, self.config.obs_dim ** 2
        self.single_observation_space = spaces.Box(low=-1, high=1, shape=(n2,), dtype=np.float16)
        self.single_action_space = spaces.Box(low=-1, high=1, shape=(self.num_modes,), dtype=np.float16)
        kw = dict(device=self.device)
        # reward | power | obs share one allocation so that a caller on the host fetches a step's results with ONE
        # device->host copy (``fetch``); the float64 arrays come first to keep them 8-byte aligned
        self._packed = torch.empty(16 * B + 2 * B * n2, dtype=torch.uint8, **kw)
        self.reward = self._packed[:8 * B].view(torch.float64)
        self.power = self._packed[8 * B:16 * B].view(torch.float64)
        self.obs = self._packed[16 * B:].view(torch.float16).view(B, n2)
        self._packed_host = None
        self.obs_f64 = torch.empty((B, n2), dtype=torch.float64, **kw)
        self.strehl = torch.zeros(B, dtype=torch.float64, **kw)
        self.ssim = torch.zeros(B, dtype=torch.float64, **kw)
        self._true = torch.ones(B, dtype=torch.bool, **kw)
        self._false = torch.zeros(B, dtype=torch.bool, **kw)
        o = _lib.AogOutputs()
        o.obs_f16, o.obs_f64 = self.obs.data_ptr(), self.obs_f64.data_ptr()
        o.reward, o.power = self.reward.data_ptr(), self.power.data_ptr()
        o.strehl, o.ssim = self.strehl.data_ptr(), self.ssim.data_ptr()
        self._out = o

    def _stream(self):
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, seed=None, options=None):
        """-> (obs, {}).  ``options={'atm_fried': r0}``: new Fried parameters from this episode on, r0 a scalar or
        ``num_envs`` values (sequence, array or tensor).  semi_dynamic draws this reset's screens at them; quasi_static
        and dynamic keep their screens, scaled per env by (r0_old / r0_new)^(5/6)."""
        if seed is not None:
            self._reseed(seed)
        self._reset_options(options)
        self._h.reset_device(self._out, self._stream())
        self._sync_counters()
        return self.obs, {}

    def step(self, actions, extrusion_noise=None):
        torch = self._torch
        if self._ssim_too_small:
            raise ValueError('win_size exceeds image extent (smf_ssim needs obs_dim^2 >= 7)')
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions), device=self.device)
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        if actions.dtype not in (torch.float32, torch.float64):
            actions = actions.to(torch.float64)
        actions = actions.contiguous()
        if actions.numel() != self.num_envs * self.num_modes:
            raise ValueError(f'actions must be [{self.num_envs}, {self.num_modes}]')
        nz_ptr = None
        if extrusion_noise is not None:
            nz = extrusion_noise
            if not torch.is_tensor(nz):
                nz = torch.as_tensor(np.asarray(nz, dtype=np.float64), device=self.device)
            nz = nz.to(self.device, torch.float64).contiguous()
            need = self.num_envs * self._h.next_extrusions() * self.num_pupil_pixels
            if nz.numel() != need:
                raise ValueError(f'extrusion_noise must have {need} elements')
            nz_ptr = nz.data_ptr() if need else None
        dt = _lib.DTYPE_F32 if actions.dtype == torch.float32 else _lib.DTYPE_F64
        done = self._h.step_device(actions.data_ptr(), dt, self._out, nz_ptr, self._stream())
        self._sync_counters()
        return self.obs, self.reward, (self._true if done else self._false), self._false, {"power": self.power}

    def fetch(self):
        """The last step's (obs float16 [B, n^2], reward float64 [B], power float64 [B]) on the host: one
        device->host copy of the packed output buffer into pinned memory, then a stream synchronise.  The returned
        tensors are views of that pinned buffer (overwritten by the next ``fetch``)."""
        torch = self._torch
        B, n2 = self.num_envs, self.config.obs_dim ** 2
        if self._packed_host is None:
            self._packed_host = torch.empty(self._packed.numel(), dtype=torch.uint8).pin_memory()
        h = self._packed_host
        h.copy_(self._packed, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return h[16 * B:].view(torch.float16).view(B, n2), h[:8 * B].view(torch.float64), h[8 * B:16 * B].view(torch.float64)

    def SH_step(self, noise='poisson', noisy_image=None):
        """Batched ``SH_step`` (AO_env.py:254-290): -> (actions [B, K] float64 cuda, ones [B] int64)."""
        torch = self._torch
        if not self.SH_operation:
            raise AttributeError("'AOVecEnv' object has no attribute 'shwfs'")
        if not hasattr(self, 'sh_action'):
            self.sh_action = torch.empty((self.num_envs, self.num_modes), dtype=torch.float64, device=self.device)
            self._ones = torch.ones(self.num_envs, dtype=torch.int64, device=self.device)
        img_ptr = None
        if noise == 'injected':
            img = torch.as_tensor(noisy_image).to(self.device, torch.float64).contiguous()
            if img.numel() != self.num_envs * self.num_pupil_pixels ** 2:
                raise ValueError('noisy_image must be [B, Np^2]')
            img_ptr = img.data_ptr()
        self._h.sh_step_device(self.sh_action.data_ptr(), noise, img_ptr, self._stream())
        return self.sh_action, self._ones

    def set_screens(self, screens):
        """[B, Np^2] torch (cuda, float32/float64) or NumPy array."""
        torch = self._torch
        if torch.is_tensor(screens) and screens.is_cuda:
            s = screens.contiguous()
            dt = _lib.DTYPE_F32 if s.dtype == torch.float32 else _lib.DTYPE_F64
            if s.dtype not in (torch.float32, torch.float64):
                raise ValueError('screens must be float32 or float64')
            self._h.set_screens_device(s.data_ptr(), dt, 0, self.num_envs)
        else:
            self._h.set_screens(np.asarray(screens))
