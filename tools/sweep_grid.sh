#!/bin/bash
# BASELINE.json configs[4], the pupil / focal grid axis on one B200: env-steps/s of the 64-actuator quasi-static
# workload (precision 'fused') at pupil 128^2 / 240^2 / 256^2 x focal 64^2 / 128^2 / 256^2 (the fused path never forms
# the focal plane, so the focal grid only changes host-side tables), pupil 512^2 x focal 128^2 / 256^2 on the fused
# kernel, and pupil 512^2 on the FP64 kernels for comparison.  Fused points also report the optics kernel's device time
# (k_dm_phase_tc, last chunk of one step, the library's timing events).  Writes the card's name and power limit, then
# one JSON line per point.
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
ENVS=${ENVS:-4096}
python - <<PY
import json, os, sys, time
sys.path.insert(0, '.')
import numpy as np, torch
from adaptive_optics_gym_b200 import AOVecEnv
kw = dict(atm_type='quasi_static', atm_fried=0.20, act_type='num_actuators', act_dim=64, obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=30)
def run(Np, Nf, B, prec, steps):
    env = AOVecEnv(B, **kw, precision=prec, seed=1, num_pupil_pixels=Np, num_focal_pixels_fiber=Nf)
    a = torch.empty((B, 64), device='cuda').uniform_(-1, 1)
    env.reset()
    for _ in range(3): env.step(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        if i % 30 == 0: env.reset()
        env.step(a)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    kernel_ms = None
    if prec == 'fused':
        env._h.set_timing(True)
        env.step(a)
        kernel_ms = round(env._h.last_kernel_ms()['field'], 4)
        env._h.set_timing(False)
    env.close()
    print(json.dumps(dict(pupil=Np, focal=Nf, envs=B, precision=prec, ms_per_step=round(ms, 4), env_steps_per_s=round(B / ms * 1e3),
                          optics_kernel_ms=kernel_ms,
                          hbm_gbs=round(4.0 * Np * Np * B / ms / 1e6, 1) if prec == 'fused' else None)), flush=True)
B = int(os.environ.get('ENVS', '4096'))
for Np in (128, 240, 256):
    for Nf in (64, 128, 256):
        run(Np, Nf, B, 'fused', 60)
run(512, 128, B, 'fused', 30)
run(512, 256, B, 'fused', 30)
run(512, 128, 256, 'f64', 6)
run(512, 256, 256, 'f64', 6)
PY
