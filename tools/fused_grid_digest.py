"""Seeded run of the fused path at one pupil / focal grid, reduced to a SHA-256 of every output it returned, to check
that two builds compute the same bits (a kernel change that must not alter results: compare the two digests).

    python tools/fused_grid_digest.py [--pupil 256] [--focal 128] [--obs-dim 5] [--envs 1000] [--steps 4]
    AOG_LIB=/path/to/other/libaogym.so python tools/fused_grid_digest.py ...       # the same run on another build

The screens come from the handle's seeded synthesis, the actions from a seeded NumPy generator; the env count is not a
multiple of 128 by default, so a partial env block is covered.  Prints one JSON line."""
import argparse
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pupil', type=int, default=256)
    ap.add_argument('--focal', type=int, default=128)
    ap.add_argument('--obs-dim', type=int, default=5)
    ap.add_argument('--envs', type=int, default=1000)
    ap.add_argument('--steps', type=int, default=4)
    ap.add_argument('--seed', type=int, default=1)
    args = ap.parse_args()
    import numpy as np
    import torch
    from adaptive_optics_gym_b200 import AOVecEnv
    kw = dict(atm_type='quasi_static', atm_fried=0.15, act_type='num_actuators', act_dim=64, obs_dim=args.obs_dim,
              rew_type='strehl_ratio', timesteps_per_episode=30)
    env = AOVecEnv(args.envs, **kw, precision='fused', seed=args.seed, num_pupil_pixels=args.pupil,
                   num_focal_pixels_fiber=args.focal)
    rng = np.random.default_rng(args.seed)
    h = hashlib.sha256()
    env.reset()
    h.update(env.obs_f64.cpu().numpy().tobytes())
    for _ in range(args.steps):
        a = torch.from_numpy(rng.uniform(-1, 1, (args.envs, 64)).astype(np.float32)).cuda()
        obs, rew, done, _, info = env.step(a)
        torch.cuda.synchronize()
        for x in (env.obs_f64, obs, rew, done, info['power'], env.strehl):
            h.update(x.cpu().numpy().tobytes())
    env.close()
    print(json.dumps(dict(pupil=args.pupil, focal=args.focal, obs_dim=args.obs_dim, envs=args.envs, steps=args.steps,
                          seed=args.seed, lib=os.environ.get('AOG_LIB', 'default'), sha256=h.hexdigest())), flush=True)


if __name__ == '__main__':
    main()
