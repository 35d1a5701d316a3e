"""ctypes binding of ``libaogym.so`` (C-ABI in ``include/aogym.h``).

There is no CPU fallback: importing this module on a machine without the built
library raises, and every entry point needs a B200.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('AOG_LIB') or os.path.join(_HERE, 'libaogym.so')   # AOG_LIB: tuning builds only

ABI_VERSION = 2

ATM = {'quasi_static': 0, 'semi_dynamic': 1, 'dynamic': 2}
REW = {'strehl_ratio': 0, 'smf_ssim': 1}
DTYPE_F32, DTYPE_F64 = 0, 1
PRECISION = {'f64': 0, 'tensor': 1, 'fused': 2}

TABLE_IDS = {
    'aperture': 0, 'dm_modes': 1, 'dm_gram': 2, 'mft_fib_1': 3, 'mft_fib_2': 4, 'mft_obs_1': 5,
    'mft_obs_2': 6, 'lp_modes_w': 7, 'lp_phase': 8, 'lp_gram': 9, 'ar_stencil': 10, 'ar_A': 11,
    'ar_B': 12, 'scr_C1': 13, 'scr_W1': 14, 'scr_C2': 15, 'scr_W2': 16,
    # Shack-Hartmann integrator (after Handle.sh_configure)
    'sh_mla_phase': 17, 'sh_fresnel': 18, 'sh_pix_offsets': 19, 'sh_pix_index': 20, 'sh_pix_x': 21,
    'sh_pix_y': 22, 'sh_offset': 23, 'sh_recon': 24, 'sh_act0': 25,
}
INT32_TABLES = ('ar_stencil', 'sh_pix_offsets', 'sh_pix_index')
SH_NOISE = {'none': 0, 'poisson': 1, 'injected': 2}
FIELD_IDS = {'screen': 0, 'pupil': 1, 'focal': 2, 'focal_power': 3, 'obs_power': 4, 'actuators': 5,
             'tc_pupil': 6, 'tc_stage1': 7, 'sh_image': 8, 'sh_actuators': 9, 'sh_image_tc': 10}


class AogConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        'abi_version', 'device', 'num_envs', 'num_pupil_pixels', 'num_focal_pixels', 'obs_dim',
        'num_modes', 'num_lp_modes', 'num_stencil', 'num_screen_fine', 'atm_type', 'rew_type',
        'sh_operation', 'flat_mirror_start', 'max_steps', 'has_rew_threshold', 'precision',
        'env_id_base')] + [(n, C.c_double) for n in (
        'rew_threshold', 'wavelength_wfs', 'wavelength_sci', 'delta_t', 'velocity', 'pupil_delta',
        'amp_fiber', 'sqrt_cn2', 'strehl_scale', 'obs_weight', 'ssim_ref_peak', 'mft_norm_re',
        'mft_norm_im')] + [('seed', C.c_uint64)]


class AogOutputs(C.Structure):
    _fields_ = [('obs_f16', C.c_void_p), ('obs_f64', C.c_void_p), ('reward', C.c_void_p),
                ('power', C.c_void_p), ('strehl', C.c_void_p), ('ssim', C.c_void_p)]


class AogCounters(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ('timestep', 'timestep_render', 'episode_no', 'column_origin',
                                         'extrusions', 'screen_draws', 'sh_draws')]


class AogError(RuntimeError):
    pass


_lib = None


def load():
    """Load libaogym.so (once).  Fails loudly when the CUDA library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(or `make -C adaptive_optics_gym_b200/csrc`).  There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    sig = {
        'aog_version': (C.c_char_p, []),
        'aog_create': (C.c_int, [C.POINTER(AogConfig), C.POINTER(P)]),
        'aog_destroy': (None, [P]),
        'aog_last_error': (C.c_char_p, [P]),
        'aog_set_table': (C.c_int, [P, C.c_int, P, C.c_size_t]),
        'aog_set_screens': (C.c_int, [P, P, C.c_int, C.c_int, C.c_int, C.c_int]),
        'aog_get_screens': (C.c_int, [P, P, C.c_int, C.c_int]),
        'aog_generate_screens': (C.c_int, [P, P]),
        'aog_next_extrusions': (C.c_int, [P]),
        'aog_set_turbulence': (C.c_int, [P, P, C.c_int, P]),
        'aog_reset': (C.c_int, [P, C.POINTER(AogOutputs), P]),
        'aog_reset_host': (C.c_int, [P, C.POINTER(AogOutputs)]),
        'aog_step': (C.c_int, [P, P, C.c_int, P, C.POINTER(AogOutputs), C.POINTER(C.c_int32), P]),
        'aog_step_host': (C.c_int, [P, P, C.c_int, P, C.POINTER(AogOutputs), C.POINTER(C.c_int32)]),
        'aog_sh_configure': (C.c_int, [P, C.c_int, C.c_int, C.c_double, C.c_double]),
        'aog_sh_step': (C.c_int, [P, C.c_int, P, P, P]),
        'aog_sh_step_host': (C.c_int, [P, C.c_int, P, P]),
        'aog_get_counters': (C.c_int, [P, C.POINTER(AogCounters)]),
        'aog_set_counters': (C.c_int, [P, C.POINTER(AogCounters)]),
        'aog_get_actuators': (C.c_int, [P, P]),
        'aog_set_actuators': (C.c_int, [P, P]),
        'aog_get_sh_actuators': (C.c_int, [P, P]),
        'aog_set_sh_actuators': (C.c_int, [P, P]),
        'aog_reseed': (C.c_int, [P, C.c_uint64]),
        'aog_health': (C.c_int, [P]),
        'aog_get_field': (C.c_int, [P, C.c_int, C.c_int, P, C.c_size_t]),
        'aog_debug_poisson': (C.c_int, [C.c_int, C.c_double, C.c_int, C.c_uint64, P]),
        'aog_debug_poisson_f32': (C.c_int, [C.c_int, C.c_double, C.c_int, C.c_uint64, P]),
        'aog_debug_normals': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, P, P, P]),
        'aog_launch_count': (C.c_int64, [P]),
        'aog_chunk_size': (C.c_int, [P]),
        'aog_set_timing': (C.c_int, [P, C.c_int]),
        'aog_last_mft_ms': (C.c_double, [P]),
        'aog_last_timings': (C.c_int, [P, C.POINTER(C.c_double), C.c_int]),
        'aog_last_kernel_ms': (C.c_int, [P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Handle:
    """Owns one ``aog_env*`` (one device, N lock-stepped environments)."""

    def __init__(self, cfg: AogConfig):
        self.lib = load()
        self._h = C.c_void_p()
        rc = self.lib.aog_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            msg = self.lib.aog_last_error(self._h).decode() if self._h else 'aog_create failed'
            if self._h:
                self.lib.aog_destroy(self._h)
                self._h = C.c_void_p()
            raise AogError(f'aog_create: {msg} (status {rc})')
        self.cfg = cfg

    def check(self, rc, what):
        if rc != 0:
            raise AogError(f'{what}: {self.lib.aog_last_error(self._h).decode()} (status {rc})')

    def close(self):
        if getattr(self, '_h', None):
            self.lib.aog_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- tables / state
    def set_table(self, name, arr):
        tid = TABLE_IDS[name]
        if name in INT32_TABLES:
            a = np.ascontiguousarray(arr, dtype=np.int32)
            count = a.size
        elif np.iscomplexobj(arr):
            a = np.ascontiguousarray(arr, dtype=np.complex128)
            count = a.size
        else:
            a = np.ascontiguousarray(arr, dtype=np.float64)
            count = a.size
        self.check(self.lib.aog_set_table(self._h, tid, _ptr(a), count), f'aog_set_table({name})')

    def set_screens(self, screens, first_env=0):
        s = np.asarray(screens)
        if s.dtype == np.float32:
            dt = DTYPE_F32
        else:
            s = s.astype(np.float64, copy=False)
            dt = DTYPE_F64
        s = np.ascontiguousarray(s).reshape(-1, self.cfg.num_pupil_pixels ** 2)
        self.check(self.lib.aog_set_screens(self._h, _ptr(s), dt, 0, first_env, s.shape[0]), 'aog_set_screens')

    def set_screens_device(self, data_ptr, dtype, first_env, count):
        self.check(self.lib.aog_set_screens(self._h, C.c_void_p(data_ptr), dtype, 1, first_env, count),
                   'aog_set_screens')

    def get_screens(self, first_env=0, count=None):
        count = self.cfg.num_envs - first_env if count is None else count
        out = np.empty((count, self.cfg.num_pupil_pixels ** 2))
        self.check(self.lib.aog_get_screens(self._h, _ptr(out), first_env, count), 'aog_get_screens')
        return out

    def generate_screens(self, stream=None):
        self.check(self.lib.aog_generate_screens(self._h, C.c_void_p(stream or 0)), 'aog_generate_screens')

    def set_turbulence(self, sqrt_cn2, rescale=False, stream=None):
        """Per-env sqrt(Cn^2) [num_envs]; ``rescale`` also multiplies each env's screen by new / old."""
        v = np.ascontiguousarray(sqrt_cn2, dtype=np.float64)
        if v.shape != (self.cfg.num_envs,):
            raise ValueError(f'sqrt_cn2 must have {self.cfg.num_envs} values')
        self.check(self.lib.aog_set_turbulence(self._h, _ptr(v), int(bool(rescale)), C.c_void_p(stream or 0)),
                   'aog_set_turbulence')

    def next_extrusions(self):
        return self.lib.aog_next_extrusions(self._h)

    def counters(self):
        c = AogCounters()
        self.check(self.lib.aog_get_counters(self._h, C.byref(c)), 'aog_get_counters')
        return c

    def set_counters(self, **kw):
        c = self.counters()
        for k, v in kw.items():
            setattr(c, k, int(v))
        self.check(self.lib.aog_set_counters(self._h, C.byref(c)), 'aog_set_counters')

    def get_actuators(self):
        out = np.empty((self.cfg.num_envs, self.cfg.num_modes))
        self.check(self.lib.aog_get_actuators(self._h, _ptr(out)), 'aog_get_actuators')
        return out

    def set_actuators(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(self.cfg.num_envs, self.cfg.num_modes)
        self.check(self.lib.aog_set_actuators(self._h, _ptr(a)), 'aog_set_actuators')

    def get_sh_actuators(self):
        out = np.empty((self.cfg.num_envs, self.cfg.num_modes))
        self.check(self.lib.aog_get_sh_actuators(self._h, _ptr(out)), 'aog_get_sh_actuators')
        return out

    def set_sh_actuators(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(self.cfg.num_envs, self.cfg.num_modes)
        self.check(self.lib.aog_set_sh_actuators(self._h, _ptr(a)), 'aog_set_sh_actuators')

    def reseed(self, seed):
        self.check(self.lib.aog_reseed(self._h, C.c_uint64(int(seed) & (2 ** 64 - 1))), 'aog_reseed')
        self.cfg.seed = int(seed) & (2 ** 64 - 1)

    def health(self):
        self.check(self.lib.aog_health(self._h), 'aog_health')

    def get_field(self, which, env_index=0):
        c = self.cfg
        P, nf2, n2 = c.num_pupil_pixels ** 2, c.num_focal_pixels ** 2, c.obs_dim ** 2
        size = {'screen': P, 'pupil': 2 * P, 'focal': 2 * nf2, 'focal_power': nf2, 'obs_power': n2,
                'actuators': c.num_modes, 'tc_pupil': 2 * P, 'sh_image': P, 'sh_image_tc': P, 'sh_actuators': c.num_modes,
                'tc_stage1': 2 * c.num_focal_pixels * c.num_pupil_pixels}[which]
        out = np.empty(size)
        self.check(self.lib.aog_get_field(self._h, FIELD_IDS[which], env_index, _ptr(out), size), 'aog_get_field')
        if which in ('pupil', 'focal', 'tc_pupil', 'tc_stage1'):
            return out.view(np.complex128)
        return out

    # ---- host-buffer step / reset (copies inside)
    def _host_outputs(self):
        B, n2 = self.cfg.num_envs, self.cfg.obs_dim ** 2
        if not hasattr(self, '_hout'):
            self._hout = dict(obs_f16=np.empty((B, n2), np.float16), obs_f64=np.empty((B, n2)),
                              reward=np.empty(B), power=np.empty(B), strehl=np.zeros(B), ssim=np.zeros(B))
            o = AogOutputs()
            for k, v in self._hout.items():
                setattr(o, k, v.ctypes.data)
            self._hout_struct = o
        return self._hout, self._hout_struct

    def reset_host(self):
        h, o = self._host_outputs()
        self.check(self.lib.aog_reset_host(self._h, C.byref(o)), 'aog_reset_host')
        return h

    def step_host_fast(self, a):
        """``step_host`` for the single-env hot loop: ``a`` is a C-contiguous float32 / float64 array of the right size,
        no extrusion noise; ctypes arguments are built once."""
        if not hasattr(self, '_fast'):
            h, o = self._host_outputs()
            done = C.c_int32(0)
            self._fast = (h, C.byref(o), done, C.byref(done), self.lib.aog_step_host)
        h, o_ref, done, done_ref, fn = self._fast
        rc = fn(self._h, a.ctypes.data, DTYPE_F32 if a.dtype == np.float32 else DTYPE_F64, None, o_ref, done_ref)
        if rc != 0:
            self.check(rc, 'aog_step_host')
        return h, done.value != 0

    def step_host(self, actions, noise=None):
        a = np.asarray(actions)
        if a.dtype == np.float32:
            dt = DTYPE_F32
        else:
            a = a.astype(np.float64, copy=False)
            dt = DTYPE_F64
        a = np.ascontiguousarray(a)
        if a.size != self.cfg.num_envs * self.cfg.num_modes:
            raise ValueError(f'actions must have {self.cfg.num_envs} x {self.cfg.num_modes} elements')
        nz = None
        if noise is not None:
            nz = np.ascontiguousarray(noise, dtype=np.float64)
            need = self.cfg.num_envs * self.next_extrusions() * self.cfg.num_pupil_pixels
            if nz.size != need:
                raise ValueError(f'noise must have {need} elements, got {nz.size}')
        h, o = self._host_outputs()
        done = C.c_int32(0)
        self.check(self.lib.aog_step_host(self._h, _ptr(a), dt, _ptr(nz), C.byref(o), C.byref(done)), 'aog_step_host')
        return h, bool(done.value)

    # ---- device-pointer step / reset (torch tensors own the buffers)
    def reset_device(self, out: AogOutputs, stream=0):
        self.check(self.lib.aog_reset(self._h, C.byref(out), C.c_void_p(stream)), 'aog_reset')

    def step_device(self, actions_ptr, act_dtype, out: AogOutputs, noise_ptr=None, stream=0):
        done = C.c_int32(0)
        self.check(self.lib.aog_step(self._h, C.c_void_p(actions_ptr), act_dtype,
                                     C.c_void_p(noise_ptr) if noise_ptr else None, C.byref(out), C.byref(done),
                                     C.c_void_p(stream)), 'aog_step')
        return bool(done.value)

    # ---- Shack-Hartmann integrator (AOEnv.SH_step)
    def sh_configure(self, num_sub, num_pix, amplitude, weight_dt):
        self.check(self.lib.aog_sh_configure(self._h, int(num_sub), int(num_pix), float(amplitude), float(weight_dt)),
                   'aog_sh_configure')

    def sh_step_host(self, noise='poisson', noisy_image=None):
        B, K, P = self.cfg.num_envs, self.cfg.num_modes, self.cfg.num_pupil_pixels ** 2
        img = None
        if noise == 'injected':
            img = np.ascontiguousarray(noisy_image, dtype=np.float64)
            if img.size != B * P:
                raise ValueError(f'noisy_image must have {B} x {P} elements')
        out = np.empty((B, K))
        self.check(self.lib.aog_sh_step_host(self._h, SH_NOISE[noise], _ptr(img), _ptr(out)), 'aog_sh_step_host')
        return out

    def sh_step_device(self, action_out_ptr, noise='poisson', noisy_image_ptr=None, stream=0):
        self.check(self.lib.aog_sh_step(self._h, SH_NOISE[noise],
                                        C.c_void_p(noisy_image_ptr) if noisy_image_ptr else None,
                                        C.c_void_p(action_out_ptr), C.c_void_p(stream)), 'aog_sh_step')

    def launch_count(self):
        return int(self.lib.aog_launch_count(self._h))

    def chunk_size(self):
        return int(self.lib.aog_chunk_size(self._h))

    def set_timing(self, on):
        self.check(self.lib.aog_set_timing(self._h, int(bool(on))), 'aog_set_timing')

    def last_kernel_ms(self):
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        self.check(self.lib.aog_last_kernel_ms(self._h, C.byref(a), C.byref(b), C.byref(c)), 'aog_last_kernel_ms')
        return dict(field=a.value, stage1=b.value, stage2=c.value)

    def last_timings(self):
        """{'extrusions_ms', 'extrusions', 'sh_phase', 'sh_fold', 'sh_gemm1', 'sh_gemm2', 'sh_camera'} of the last
        timed step (ms; -1 = not recorded)"""
        buf = (C.c_double * 7)()
        self.check(self.lib.aog_last_timings(self._h, buf, 7), 'aog_last_timings')
        names = ('extrusions_ms', 'extrusions', 'sh_phase', 'sh_fold', 'sh_gemm1', 'sh_gemm2', 'sh_camera')
        return dict(zip(names, (float(v) for v in buf)))

    def last_mft_ms(self):
        return float(self.lib.aog_last_mft_ms(self._h))
