#!/usr/bin/env python
"""bench.py -- env-steps/sec of the AO-v0 step path on N B200s (one JSON line on rank 0).

A "step" is one lock-stepped ``AOVecEnv.step`` over the rank's batch of environments (B env-steps),
including the ``reset`` at every episode boundary (the timed window is phased so that it always holds at least one)
and the end-of-episode ``gather_episode_stats`` (the one collective of the design: NCCL all-reduce of the episode
returns).  Headline workload (BASELINE.json: "64-act quasi-static"): quasi_static, r0 = 0.20 m, 64 disk-harmonic
actuators, 2x2 photodetector, strehl_ratio reward, 30 steps/episode (configs[0] physics), batched at ``--envs``
environments per GPU (weak scaling).

  value      device-resident throughput: actions already in HBM, outputs left in HBM
  e2e        same metric through the public API with HOST buffers: pinned host actions copied host->device every
             step, obs/reward/power copied device->host every step
  roofline   the dominant kernel timed live with CUDA events on the launch stream inside the library
  workloads  the other BASELINE.json configs (configs[1..3]) in short runs: value, ms_per_step, dominant kernel and its
             roofline fraction -- under torchrun too, so the scaling record carries them at 1/2/4/8 GPUs
  cpu_baseline  the CPU oracle (NumPy FP64, unabridged reference op sequence) on this box's cores: single env with the
             default BLAS threads (value), with one thread, and one single-thread env per core in parallel

``--impl reference`` times the reference-side CPU implementation (the oracle port; hcipy itself is not installable
here) on the host cores for the same metric / config, using every host thread: one single-thread env per core.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json metric config: 64-actuator quasi-static (configs[0] physics), batched
    'quasi_static_64act': dict(atm_type='quasi_static', atm_vel=0, atm_fried=0.20, act_type='num_actuators',
                               act_dim=64, obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=30,
                               flat_mirror_start_per_episode=True),
    # BASELINE.json configs[1]
    'zernike6_smf_ssim': dict(atm_type='quasi_static', atm_vel=0, atm_fried=0.15, act_type='zernike', act_dim=6,
                              obs_dim=5, rew_type='smf_ssim', timesteps_per_episode=20,
                              flat_mirror_start_per_episode=True),
    # BASELINE.json configs[2] as the reference runs it: semi_dynamic coerces the velocity to 0 (AO_env.py:200-203) and
    # draws a fresh von-Karman screen at every reset (:76-77)
    'semi_dynamic_64act': dict(atm_type='semi_dynamic', atm_vel=0, atm_fried=0.15, act_type='num_actuators', act_dim=64,
                               obs_dim=5, rew_type='strehl_ratio', timesteps_per_episode=20,
                               flat_mirror_start_per_episode=True),
    # ... and with the phase-screen evolution that config names (dynamic, 5 m/s: 2.4 extrusions per step)
    'dynamic_v5': dict(atm_type='dynamic', atm_vel=5, atm_fried=0.15, act_type='num_actuators', act_dim=64,
                       obs_dim=5, rew_type='strehl_ratio', timesteps_per_episode=20,
                       flat_mirror_start_per_episode=True),
    # BASELINE.json configs[3] physics without the SH loop
    'dynamic_v20': dict(atm_type='dynamic', atm_vel=20, atm_fried=0.10, act_type='num_actuators', act_dim=64,
                        obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=20,
                        flat_mirror_start_per_episode=True),
    # BASELINE.json configs[3]: the Shack-Hartmann integrator drives the mirror (SH_step + step every step)
    'dynamic_v20_sh': dict(atm_type='dynamic', atm_vel=20, atm_fried=0.10, act_type='num_actuators', act_dim=64,
                           obs_dim=2, rew_type='strehl_ratio', timesteps_per_episode=20,
                           flat_mirror_start_per_episode=True, SH_operation=True),
}
# the extra workloads of the default run: (name, total envs over all GPUs or None = --envs per GPU)
EXTRA = [('zernike6_smf_ssim', None), ('semi_dynamic_64act', 16384), ('dynamic_v5', None), ('dynamic_v20', None),
         ('dynamic_v20_sh', None)]

MFT_FLOP_PER_ENV = lambda Np, Nf: 8.0 * (Nf * Np * Np + Nf * Np * Nf)   # SURVEY 8(d): 90.44 MFLOP @ 240/128
EXTRUSION_FLOP = lambda Np, Ns: 2.0 * Np * (Ns + Np)                    # SURVEY 8(d): 0.4608 MFLOP @ 240 / 720
FP64_PEAK_TFLOPS = 37.0   # nominal B200 FP64 (MEASURED_PEAKS.json has no FP64 figure)


def describe(name, envs, n_gpus):
    w = WORKLOADS[name]
    return (f"{w['atm_type']} r0={w['atm_fried']} {w['act_type']} K={w['act_dim']} obs {w['obs_dim']}x{w['obs_dim']} "
            f"{w['rew_type']} {w['timesteps_per_episode']} steps/episode, {envs} envs/GPU x {n_gpus} GPU")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.rows = []
        self.stop_flag = threading.Event()
        self.index = index

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-i',
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(int(float(r[0])) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        try:
            mx = int(float(self.rows[0][1]))
        except ValueError:
            mx = None
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': reasons,
                'samples': len(self.rows)}


# ---------------------------------------------------------------------------------------------- CPU side
def cpu_episode_rates(name, episodes, warmup_episodes=1):
    """steps/s of each of `episodes` episodes of the CPU oracle (single env, the reference's own shape),
    after `warmup_episodes`: BASELINE.md 4.3 protocol (actions ~ U(-1, 1) float32 seed 1, screen seed 0)."""
    import numpy as np
    from oracle.ao_oracle import OracleAOEnv
    w = WORKLOADS[name]
    env = OracleAOEnv(**w, seed=0)
    rng = np.random.default_rng(1)
    K, T = w['act_dim'], w['timesteps_per_episode']
    sh = bool(w.get('SH_operation'))

    def episode():
        env.reset()
        for _ in range(T):
            env.step(env.SH_step()[0] if sh else rng.uniform(-1, 1, K).astype(np.float32))

    for _ in range(warmup_episodes):
        episode()
    rates = []
    for _ in range(episodes):
        t0 = time.perf_counter()
        episode()
        rates.append(T / (time.perf_counter() - t0))
    return rates


def cpu_worker(args):
    """one single-thread CPU env (spawned by `parallel_cpu_rate`): prints its env-steps/s over --steps episodes"""
    rates = cpu_episode_rates(args.workload, args.steps, max(args.warmup, 1))
    T = WORKLOADS[args.workload]['timesteps_per_episode']
    print(json.dumps({'rate': len(rates) * T / sum(T / r for r in rates), 'episodes': len(rates)}), flush=True)


def parallel_cpu_rate(name, procs, episodes, warmup=1):
    """`procs` independent single-thread CPU envs side by side (how the reference uses every core: it has no batching)"""
    env = dict(os.environ)
    for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        env[k] = '1'
    cmd = [sys.executable, os.path.abspath(__file__), '--cpu-worker', '--workload', name, '--steps', str(episodes),
           '--warmup', str(warmup)]
    ps = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env) for _ in range(procs)]
    total = 0.0
    for p in ps:
        out, _ = p.communicate(timeout=600)
        total += json.loads(out.strip().splitlines()[-1])['rate']
    return total


def cpu_baseline(name, episodes=10):
    """BASELINE.md 4.3: median over 10 episodes after one warm-up episode, with the default BLAS threads and with one
    thread; plus one single-thread env per core side by side (the fairest use of the box for an unbatched env)."""
    import numpy as np
    from threadpoolctl import threadpool_limits
    cores = os.cpu_count()
    T = WORKLOADS[name]['timesteps_per_episode']
    default = float(np.median(cpu_episode_rates(name, episodes)))
    with threadpool_limits(limits=1):
        single = float(np.median(cpu_episode_rates(name, episodes)))
    par = parallel_cpu_rate(name, cores, 4)
    return {'value': default, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
            'sample': f'median of {episodes} episodes x {T} steps of one env after 1 warm-up episode, NumPy/OpenBLAS '
                      'default threads, unabridged reference op sequence (oracle port; hcipy==0.5.1 not installable)',
            'single_thread': {'value': single, 'unit': 'env-steps/s', 'threads': 1},
            'parallel_single_thread_envs': {'value': par, 'unit': 'env-steps/s', 'processes': cores,
                                            'sample': f'{cores} processes x 4 episodes, OMP_NUM_THREADS=1 each'}}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    # The reference has no batching: the way it uses every host thread is one single-thread env per core.  One bench
    # "step" = one episode on every one of those envs.
    cores = int(os.environ.get('AOG_REF_THREADS', str(os.cpu_count())))
    w = WORKLOADS[args.workload]
    T = w['timesteps_per_episode']
    t0 = time.perf_counter()
    v = parallel_cpu_rate(args.workload, cores, args.steps, max(args.warmup, 1))
    wall = time.perf_counter() - t0
    line = {
        'impl': 'reference', 'metric': 'env-steps/sec', 'value': v, 'unit': 'env-steps/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * cores * T / v, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': describe(args.workload, args.envs, args.gpus),
                   'note': f'reference arm = {cores} independent single-thread CPU envs side by side (the reference has '
                           f'no batching); one bench step = one {T}-step episode incl. reset on every env'},
        'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{cores} processes x {args.steps} episodes x {T} steps, NumPy/OpenBLAS 1 thread each '
                                   f'(hcipy==0.5.1 is not installable here: oracle port, unabridged op sequence); '
                                   f'{wall:.0f} s wall incl. set-up'},
        'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- GPU side
class Runner:
    """One AOVecEnv driven episode by episode: reset at every episode boundary, returns accumulated on the device,
    gather_episode_stats (NCCL all-reduce) at every episode end."""

    def __init__(self, name, B, local, rank, precision, seed=1234):
        import torch
        from adaptive_optics_gym_b200 import AOVecEnv
        self.torch = torch
        self.w = WORKLOADS[name]
        self.B, self.K, self.T = B, self.w['act_dim'], self.w['timesteps_per_episode']
        self.dev = torch.device('cuda', local)
        self.env = AOVecEnv(B, **self.w, device=local, seed=seed, precision=precision, env_id_base=rank * B)
        g = torch.Generator(device='cpu').manual_seed(7 + rank)
        self.pool = 8
        self.act_host = [torch.empty((B, self.K), dtype=torch.float32).uniform_(-1, 1, generator=g).pin_memory()
                         for _ in range(self.pool)]
        self.act_dev = [a.to(self.dev) for a in self.act_host]
        self.sh_loop = bool(self.w.get('SH_operation'))
        self.ret = torch.zeros(B, dtype=torch.float64, device=self.dev)
        self.t = 0
        self.resets = 0
        from adaptive_optics_gym_b200.sharding import gather_episode_stats
        self.stats = gather_episode_stats(self.ret)      # loads torch's reduction kernels / NCCL channels before any clock runs

    def _begin(self):
        if self.t % self.T == 0:
            self.env.reset()
            self.ret.zero_()
            self.resets += 1

    def _end(self, reward):
        from adaptive_optics_gym_b200.sharding import gather_episode_stats
        self.ret.add_(reward)
        self.t += 1
        if self.t % self.T == 0:
            self.stats = gather_episode_stats(self.ret)      # the design's one collective (NCCL when world > 1)

    def step_device(self, i):
        self._begin()
        a = self.env.SH_step()[0] if self.sh_loop else self.act_dev[i % self.pool]
        _, rew, self.done, _, _ = self.env.step(a)
        self._end(rew)

    def outputs(self):
        """What the last ``step_device`` handed its caller, on the host: float16 obs widened to float32, the done mask
        as 0 / 1, the Shack-Hartmann action when the integrator drives the mirror."""
        e = self.env
        out = {'obs': e.obs.float(), 'obs_f64': e.obs_f64, 'reward': e.reward, 'power': e.power,
               'done': self.done.float()}
        if self.sh_loop:
            out['sh_action'] = e.sh_action
        return {k: v.cpu().numpy() for k, v in out.items()}

    def step_e2e(self, i):
        self._begin()
        a = self.act_host[i % self.pool].to(self.dev, non_blocking=True)
        if self.sh_loop:
            a = self.env.SH_step()[0]
        _, rew, _, _, _ = self.env.step(a)
        self.env.fetch()                 # obs, reward, power -> pinned host memory (one copy) + stream synchronise:
        self._end(rew)                   # the caller needs the result before acting again

    def phase_window(self, steps, warmup):
        """Start the clock of the episode so that an episode boundary (done -> gather -> reset) falls in the middle of
        the timed window whatever --steps / --warmup are."""
        pre = (self.T - (warmup + max(steps // 2, 1))) % self.T
        self.env.reset()
        self.ret.zero_()
        self.env._h.set_counters(timestep_render=pre)
        self.t = pre if pre else self.T          # pre == 0: a reset is due at the first warm-up step


def timed(r, fn, steps, warmup, world, dist):
    import torch
    r.phase_window(steps, warmup)
    for i in range(warmup):
        fn(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0, r0 = r.env._h.launch_count(), r.resets
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = r.env._h.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=r.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, launches, r.resets - r0


DUMP_LIMIT = 64 * 10 ** 6     # bytes written by --dump-outputs, .npy headers included


def dump_outputs(arrays, out_dir):
    """Write each [B, ...] array as out_dir/<name>.npy.  When they would exceed DUMP_LIMIT, every array keeps the same
    fixed, seeded sample of env rows, whose indices go to env_index.npy."""
    import numpy as np
    B = len(next(iter(arrays.values())))
    row = sum(a.nbytes for a in arrays.values()) // B
    if B * row > DUMP_LIMIT - 4096:
        keep = np.sort(np.random.default_rng(0).choice(B, (DUMP_LIMIT - 4096) // (row + 8), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays['env_index'] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def kernel_times(r, prec, n=6):
    """median per-kernel milliseconds of one step (CUDA events on the launch stream inside the library)"""
    import torch
    e = r.env
    e._h.set_timing(True)
    mft_ms, kms, tms = [], [], []
    for i in range(n):      # no reset inside this loop
        e.step(e.SH_step()[0] if r.sh_loop else r.act_dev[i % r.pool])
        torch.cuda.synchronize()
        mft_ms.append(e._h.last_mft_ms())
        if prec != 'f64':
            kms.append(e._h.last_kernel_ms())
        tms.append(e._h.last_timings())
    e._h.set_timing(False)
    med = lambda xs: sorted(xs)[len(xs) // 2]
    km = {k: med([d[k] for d in kms[1:]]) for k in kms[0]} if kms else None
    tm = {k: med([d[k] for d in tms[1:]]) for k in tms[0]}
    return med(mft_ms[1:]), km, tm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=300)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--envs', type=int, default=4096, help='environments per GPU')
    ap.add_argument('--workload', default='quasi_static_64act', choices=list(WORKLOADS))
    ap.add_argument('--precision', default='auto', choices=['auto', 'f64', 'tensor', 'fused'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-mft-arm', action='store_true', help='skip the secondary timing of the tensor-core MFT path')
    ap.add_argument('--no-workloads', action='store_true', help='skip the short runs of the other BASELINE configs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step returned (rank 0\'s envs) as DIR/<name>.npy, to compare builds '
                         'output for output: the inputs depend only on the arguments')
    ap.add_argument('--cpu-worker', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_worker:
        return cpu_worker(args)
    if args.warmup < 3:
        args.warmup = 3
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    w = WORKLOADS[args.workload]
    B, K, n2, T = args.envs, w['act_dim'], w['obs_dim'] ** 2, w['timesteps_per_episode']
    precision = 'fused' if args.precision == 'auto' else args.precision
    run = Runner(args.workload, B, local, rank, precision)
    env = run.env
    Np, Nf = env.num_pupil_pixels, env.num_focal_pixels_fiber

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, resets = timed(run, run.step_device, args.steps, args.warmup, world, dist)
    outputs = run.outputs() if args.dump_outputs and rank == 0 else None
    value = world * B * args.steps / (ms * 1e-3)
    ms_e2e, _, _ = timed(run, run.step_e2e, args.steps, args.warmup, world, dist)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    clocks = sampler.summary() if sampler else None      # sampled over both timed regions

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = peaks.get('hbm_gbs', 6500.0)
    hbm_note = 'measured copy bandwidth (MEASURED_PEAKS.json)' if peaks else 'fallback 6.5 TB/s (B200_PROFILING.md)'

    def traffic_from_profiles(name, last_chunk):
        # dram__bytes_read + dram__bytes_write per launch from the committed ncu --set full capture (profiles/),
        # valid for the chunk size it was taken at
        try:
            tj = json.load(open(os.path.join(ROOT, 'profiles', name)))
            if tj.get('envs_per_launch') == last_chunk:
                return tj['bytes_per_launch']
        except Exception:
            pass
        return None

    def last_chunk_of(r):
        chunk = min(r.env._h.chunk_size(), r.B)
        return r.B - (r.B - 1) // chunk * chunk

    def mft_roofline(r, prec):
        """the matrix-Fourier-transform GEMMs against the tensor (or FP64) pipe"""
        mft, km, _ = kernel_times(r, prec)
        lc = last_chunk_of(r)
        achieved = MFT_FLOP_PER_ENV(Np, Nf) * lc / (mft * 1e-3) / 1e12
        if prec == 'tensor':
            peak = peaks.get('bf16_tflops_sustained', 1400.0)
            peak_note = ('measured cuBLAS bf16 sustained (MEASURED_PEAKS.json)' if peaks else
                         'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)')
            issued = 3.0
        else:
            peak = FP64_PEAK_TFLOPS
            peak_note = 'nominal B200 FP64 37 TFLOP/s (no measured FP64 peak in MEASURED_PEAKS.json)'
            issued = 1.0
        rl = {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
              'traffic': traffic_from_profiles('mft_dram_traffic.json', lc) if prec == 'tensor' else None,
              'kernel': ('matrix Fourier transform: k_field_mft1 (field formation + stage-1 product) + k_mft2 (stage-2 '
                         'product + fibre projection)') if prec == 'tensor' else 'MFT stage-1 + stage-2 complex GEMMs (FP64)',
              'ms_per_launch': mft, 'envs_per_launch': lc, 'algorithmic_flop_per_env': MFT_FLOP_PER_ENV(Np, Nf),
              'issued_over_algorithmic': issued, 'peak_source': peak_note}
        if km:
            rl['kernel_ms'] = km
        return rl

    def fused_roofline(r, km=None):
        # dominant kernel: k_dm_phase_tc<fused> -- DM-surface GEMM (tcgen05) + phase + every reduction of the step.
        # Algorithmic bytes (SURVEY 8d, fused design): one FP32-sized read of the screen per env-step, 4 P bytes.
        if km is None:
            _, km, _ = kernel_times(r, 'fused')
        lc = last_chunk_of(r)
        alg_bytes = 4.0 * Np * Np
        ach = alg_bytes * lc / (km['field'] * 1e-3) / 1e9
        return {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                'traffic': traffic_from_profiles('fused_dram_traffic.json', lc),
                'kernel': 'k_dm_phase_tc<fused>: tcgen05 DM-surface GEMM, wavefront phase, obs-arm / Strehl / '
                          'back-projected fibre-mode reductions (the whole optics chain of a step)',
                'ms_per_launch': km['field'], 'envs_per_launch': lc, 'algorithmic_bytes_per_env': alg_bytes,
                'peak_source': hbm_note,
                'note': 'the kernel is issue / SFU bound (4 MUFU per lit pixel), not HBM bound; see DESIGN.md 4.3'}

    def dominant_roofline(r, name, prec, ms_step):
        """dominant kernel of a workload's step and its roofline fraction (kernel times from the library's events)"""
        if prec != 'fused':
            return mft_roofline(r, prec)
        _, km, tm = kernel_times(r, prec)
        lc = last_chunk_of(r)
        n_chunks = -(-r.B // min(r.env._h.chunk_size(), r.B))
        cands = {'optics': km['field'] * n_chunks}          # km: the last chunk's launch; a step launches one per chunk
        if tm['extrusions'] > 0:
            cands['extrusion'] = tm['extrusions_ms']
        sh = {k: tm[k] for k in ('sh_phase', 'sh_fold', 'sh_gemm1', 'sh_gemm2', 'sh_camera') if tm[k] > 0}
        cands.update(sh)
        if WORKLOADS[name]['atm_type'] == 'semi_dynamic':       # a new von-Karman screen per episode (AO_env.py:76-77)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r.env.reset()
            e1.record()
            torch.cuda.synchronize()
            cands['reset_per_step'] = e0.elapsed_time(e1) / r.T
        top = max(cands, key=cands.get)
        if top == 'optics':
            rl = fused_roofline(r, km)
        elif top == 'reset_per_step':
            # the reset = von-Karman synthesis (DESIGN.md 4.6: the fine scale as a 240 x 240 inverse FFT whose row kernel
            # draws its normals and whose column kernel writes screens + phase tiles; the coarse scale as five small FP64
            # tensor-core GEMMs) + one optics pass.  HBM-bound by design; algorithmic bytes per env: the FFT intermediate
            # written and read (2 x 16 P), the screen written by the coarse scale, read and rewritten by the column
            # kernel (3 x 8 P), the phase tiles (4 P), the optics pass (4 P)
            alg = (32.0 + 24.0 + 4.0 + 4.0) * Np * Np
            ms_reset = cands[top] * r.T
            ach = alg * r.B / (ms_reset * 1e-3) / 1e9
            rl = {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                  'traffic': None, 'kernel': 'reset: von-Karman screen synthesis (k_scr_fft_rows + k_scr_fft_cols, coarse scale '
                                             'on the FP64 tensor cores) + the optics chain',
                  'ms_per_launch': ms_reset, 'envs_per_launch': r.B, 'algorithmic_bytes_per_env': alg,
                  'peak_source': hbm_note}
        elif top == 'extrusion':
            n_ext = tm['extrusions']
            per = tm['extrusions_ms'] / n_ext
            Ns = int(r.env.tables['ar_stencil'].size)
            ach = EXTRUSION_FLOP(Np, Ns) * r.B / (per * 1e-3) / 1e12     # every chunk is inside the timed span
            rl = {'bound': 'tensor', 'achieved': ach, 'peak': FP64_PEAK_TFLOPS, 'unit': 'TFLOP/s',
                  'frac': ach / FP64_PEAK_TFLOPS, 'traffic': None,
                  'kernel': 'k_ar_step<DIRECT>: one column extrusion new = A z + B xi for every env, stencil read in place (FP64 tensor cores)',
                  'ms_per_launch': per, 'launches_per_step': n_ext, 'envs_per_launch': r.B,
                  'algorithmic_flop_per_env': EXTRUSION_FLOP(Np, Ns),
                  'peak_source': 'nominal B200 FP64 37 TFLOP/s (no measured FP64 peak in MEASURED_PEAKS.json)'}
        else:
            # tensor-core Shack-Hartmann step (sh_tensor.cuh); algorithmic bytes per env of each kernel (no padding):
            # phase 4 P read + 4 N_ap-ish written (counted 4 P); fold 4 P read + 8 P written (4 blocks x re, im x hi, lo x
            # fp16 over P / 4 fold pixels = 8 P); products: 8 P read + 8 P written; camera: 8 P read (FP32 planes)
            P = Np * Np
            alg = {'sh_phase': 8.0 * P, 'sh_fold': 12.0 * P, 'sh_gemm1': 16.0 * P, 'sh_gemm2': 16.0 * P, 'sh_camera': 8.0 * P}[top]
            ach = alg * lc / (cands[top] * 1e-3) / 1e9
            rl = {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak, 'traffic': None,
                  'kernel': {'sh_phase': 'k_dm_phase_tc<phase only>', 'sh_fold': 'k_sh_fold', 'sh_gemm1': 'k_sh_gemm<1> (Y = C E, tcgen05)',
                             'sh_gemm2': 'k_sh_gemm<2> (G = Y C^T, tcgen05)', 'sh_camera': 'k_sh_camera_tc'}[top],
                  'ms_per_launch': cands[top], 'envs_per_launch': lc, 'algorithmic_bytes_per_env': alg, 'peak_source': hbm_note,
                  'sh_kernel_ms': sh}
        rl['step_kernel_ms'] = {k: round(v, 4) for k, v in cands.items()}
        return rl

    mft_arm = None
    if precision == 'fused':
        roofline = fused_roofline(run)
    else:
        roofline = mft_roofline(run, precision)
    if precision == 'fused' and not args.no_mft_arm and args.workload != 'dynamic_v20_sh':
        # BASELINE.json's metric also asks for the MFT tensor-pipe utilisation: time the path that runs the
        # fibre-arm matrix Fourier transform as tcgen05 GEMMs (precision='tensor') on the same workload
        rt = Runner(args.workload, B, local, rank, 'tensor')
        n_t = max(10, args.steps // 10)
        ms_t, _, _ = timed(rt, rt.step_device, n_t, 3, world, dist)
        mft_arm = {'precision': 'tensor', 'value': world * B * n_t / (ms_t * 1e-3), 'unit': 'env-steps/s',
                   'ms_per_step': ms_t / n_t, 'steps': n_t, 'roofline': mft_roofline(rt, 'tensor')}
        rt.env.close()
        del rt

    episode_stats = run.stats
    workloads = None
    if not args.no_workloads and args.workload == 'quasi_static_64act':
        env.close()
        del run, env
        torch.cuda.empty_cache()
        workloads = {}
        for name, total in EXTRA:
            ww = WORKLOADS[name]
            Bw = B if total is None else max(total // world, 1)
            rw = Runner(name, Bw, local, rank, precision)
            nst = ww['timesteps_per_episode'] + 4            # a whole episode and its reset inside the window
            ms_w, launches_w, resets_w = timed(rw, rw.step_device, nst, 3, world, dist)
            rl = dominant_roofline(rw, name, precision, ms_w / nst)
            workloads[name] = {'value': world * Bw * nst / (ms_w * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': ms_w / nst,
                               'steps': nst, 'envs_per_gpu': Bw, 'scaling': 'weak' if total is None else 'strong',
                               'resets_in_window': resets_w, 'gpu_launches': int(launches_w),
                               'workload': describe(name, Bw, world), 'dominant_kernel': rl['kernel'],
                               'roofline_frac': rl['frac'], 'roofline': rl, 'episode_stats': rw.stats}
            rw.env.close()
            del rw
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline(args.workload)

    line = {
        'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None,
        'dtype': {'f64': 'f64', 'tensor': 'f16x3(tcgen05)+f32/f64', 'fused': 'f16x3(tcgen05 DM GEMM)+f32/f64'}[precision],
        'data': 'synthetic',
        'config': {'workload': describe(args.workload, B, world), 'precision': precision, 'envs_per_gpu': B,
                   'l2_policy': (f'inputs larger than L2: {B * Np * Np * 4 / 1e6:.0f} MB of phase-screen tiles read per step, '
                                 f'plus {B * Np * Np * 4 / 1e6:.0f} MB of phase and {B * 128 * 480 * 4 / 1e6:.0f} MB of stage-1 product '
                                 'written and re-read (126 MB L2)') if precision == 'tensor' else
                                (f'inputs larger than L2: {B * Np * Np * 4 / 1e6:.0f} MB of phase-screen tiles read per step '
                                 '(126 MB L2)') if precision == 'fused' else
                                f'inputs larger than L2: {B * Np * Np * 8 / 1e6:.0f} MB of screens read per step',
                   'timing': 'CUDA events on the launch stream, max over ranks; the window is phased to hold an episode '
                             'end (gather_episode_stats all-reduce) and the reset that follows',
                   'resets_in_window': resets},
        'e2e': {'value': e2e, 'unit': 'env-steps/s', 'h2d_bytes_per_step': world * B * K * 4,
                'd2h_bytes_per_step': world * B * (n2 * 2 + 16), 'ms_per_step': ms_e2e / args.steps},
        'gpu_launches': int(launches),
        'roofline': roofline,
        'cpu_baseline': cpu,
        'clocks': clocks,
        'episode_stats': episode_stats,
    }
    if mft_arm:
        line['mft_gemm_path'] = mft_arm
    if workloads:
        line['workloads'] = workloads
    if outputs:
        dump_outputs(outputs, args.dump_outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
