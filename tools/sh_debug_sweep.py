"""Per-kernel times of the tensor-core Shack-Hartmann step (aog_last_timings) under AOG_SH_DEBUG:
which part of k_sh_gemm costs what (bits: 1 no MMA, 4 no epilogue work)."""
import os, sys, torch
sys.path.insert(0, '.')
from adaptive_optics_gym_b200 import AOVecEnv
kw = dict(atm_type='dynamic', atm_vel=20, atm_fried=0.10, act_dim=64, obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=20, SH_operation=True, seed=3)
env = AOVecEnv(4096, **kw, precision='fused')
env.reset()
for _ in range(3): env.SH_step()
env._h.set_timing(True)
for _ in range(3):
    env.SH_step(); torch.cuda.synchronize()
t = env._h.last_timings()
print(os.environ.get('AOG_SH_DEBUG', '0'), {k: round(v, 3) for k, v in t.items() if k.startswith('sh_')}, flush=True)
