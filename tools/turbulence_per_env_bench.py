#!/usr/bin/env python
"""Cost of the per-env Fried parameter (profiles/r8_turbulence_per_env.md).  Prints JSON lines and writes them to --out.

  scalar    steps/s of the scalar-r0 workloads that run the synthesis / extrusion kernels (semi_dynamic_64act,
            dynamic_v20) and the headline (quasi_static_64act), this checkout against --baseline-root (another built
            checkout, imported under another module name), alternated run by run; plus a bitwise comparison of the two
            builds' outputs and screens on a seeded run
  mixed     steps/s with r0 log-uniform in [0.05, 0.20] per env against one scalar r0 (semi_dynamic_64act, dynamic_v5)
  rescale   device time of aog_set_turbulence(rescale=1) (the pass behind reset(options={'atm_fried': ...})) on a
            quasi_static handle, against the bytes it must move
  phase     the largest |S| / lambda_wfs of the device-generated screens, scaled to r0 = 0.20 m (tables.FRIED_MIN)

    python tools/turbulence_per_env_bench.py [--envs 4096] [--steps 200] [--reps 3] [--baseline-root DIR] [--out F]
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7     # B200 data sheet, one GPU


def load_package(root, name):
    """the adaptive_optics_gym_b200 package of checkout ``root`` as module ``name`` (its own libaogym.so)"""
    pkg = os.path.join(root, 'adaptive_optics_gym_b200')
    spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, '__init__.py'),
                                                  submodule_search_locations=[pkg])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return importlib.import_module(name + '.env')


def steps_per_s(env, acts, steps, warmup):
    """env-steps/s over ``steps`` steps with a reset at every episode boundary (semi_dynamic: a new screen)"""
    import torch
    T = env.max_steps
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
            ev[0].record()
        if i % T == 0:
            env.reset()
        env.step(acts[i % len(acts)])
    ev[1].record()
    torch.cuda.synchronize()
    return env.num_envs * steps / (ev[0].elapsed_time(ev[1]) * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=25)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--baseline-root', default=None)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from bench import WORKLOADS
    from adaptive_optics_gym_b200 import env as new_env
    builds = {'new': new_env}
    if args.baseline_root:
        builds['baseline'] = load_package(os.path.abspath(args.baseline_root), 'aog_baseline')
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({'kind': 'device', 'torch_name': torch.cuda.get_device_name(0), 'nvidia_smi': q[0] if q else None})
    B = args.envs
    g = torch.Generator(device='cpu').manual_seed(7)
    acts = [torch.empty((B, 64), dtype=torch.float32).uniform_(-1, 1, generator=g).cuda() for _ in range(8)]

    # ---- scalar path: this build against the baseline, alternated
    for name in ('semi_dynamic_64act', 'dynamic_v20', 'quasi_static_64act'):
        w = WORKLOADS[name]
        envs = {k: m.AOVecEnv(B, **w, seed=1234, precision='fused') for k, m in builds.items()}
        rates = {k: [] for k in envs}
        for r in range(args.reps):
            for k in (list(envs) if r % 2 == 0 else list(envs)[::-1]):
                rates[k].append(steps_per_s(envs[k], acts, args.steps, args.warmup))
        same = None
        if len(envs) == 2:
            out = {}
            for k, e in envs.items():
                e.close()
                e = envs[k] = builds[k].AOVecEnv(B, **w, seed=99, precision='fused')
                for i in range(w['timesteps_per_episode'] + 3):     # across an episode boundary
                    if i % w['timesteps_per_episode'] == 0:
                        e.reset()
                    e.step(acts[i % 8])
                torch.cuda.synchronize()
                out[k] = [e.obs.cpu().numpy().view(np.uint16), e.reward.cpu().numpy(), e.power.cpu().numpy(),
                          e._h.get_screens(0, 64), e._h.get_screens(B - 64, 64)]
            same = all(np.array_equal(a, b) for a, b in zip(out['new'], out['baseline']))
        emit({'kind': 'scalar', 'workload': name, 'envs': B, 'steps_per_s': rates, 'bitwise_equal_outputs': same})
        for e in envs.values():
            e.close()

    # ---- a mixed batch against one scalar r0 (this build)
    rng = np.random.default_rng(0)
    r0_mix = np.exp(rng.uniform(np.log(0.05), np.log(0.20), B))
    for name in ('semi_dynamic_64act', 'dynamic_v5'):
        w = dict(WORKLOADS[name])
        envs = {'scalar': new_env.AOVecEnv(B, **w, seed=1234, precision='fused')}
        w['atm_fried'] = r0_mix
        envs['mixed'] = new_env.AOVecEnv(B, **w, seed=1234, precision='fused')
        rates = {k: [] for k in envs}
        for r in range(args.reps):
            for k in (list(envs) if r % 2 == 0 else list(envs)[::-1]):
                rates[k].append(steps_per_s(envs[k], acts, args.steps, args.warmup))
        if name == 'semi_dynamic_64act':     # screens drawn at each env's r0 (two draws: construction and resets)
            s = envs['mixed']._h.get_screens(0, 512)
            at_020 = np.abs(s).max(axis=1) * (r0_mix[:512] / 0.20) ** (5 / 6) / envs['mixed'].wavelength_wfs
            emit({'kind': 'phase', 'envs': 512, 'max_abs_S_over_lambda_wfs_at_r0_0.20_rad': float(at_020.max()),
                  'median_rad': float(np.median(at_020))})
        emit({'kind': 'mixed', 'workload': name, 'envs': B, 'r0': 'log-uniform [0.05, 0.20]', 'steps_per_s': rates})
        for e in envs.values():
            e.close()

    # ---- the rescale pass: screens read + written (FP64), phase tiles written (int32)
    w = WORKLOADS['quasi_static_64act']
    e = new_env.AOVecEnv(B, **w, seed=1234, precision='fused')
    e.reset()
    from adaptive_optics_gym_b200.tables import sqrt_cn2_from_fried
    vals = [sqrt_cn2_from_fried(r, e.wavelength_sci) for r in (r0_mix, r0_mix[::-1].copy())]
    stream = e._stream()
    for i in range(5):
        e._h.set_turbulence(vals[i % 2], True, stream)
    n = 40
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for i in range(n):
        e._h.set_turbulence(vals[i % 2], True, stream)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / n
    P = e.num_pupil_pixels ** 2
    nbytes = B * P * (8 + 8 + 4)
    emit({'kind': 'rescale', 'envs': B, 'ms_per_call': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms * 1e-6,
          'hbm_floor_ms': nbytes / (HBM_TBPS * 1e12) * 1e3, 'share_of_hbm_datasheet': nbytes / (HBM_TBPS * 1e12) * 1e3 / ms})
    e.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            for d in lines:
                f.write(json.dumps(d) + '\n')


if __name__ == '__main__':
    main()
