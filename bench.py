#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched BabyAI pool (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--level L] [--envs E] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- BabyAI-GoToLocal-v0,
65 536 environments per GPU, uniform random actions, ParallelEnv auto-reset on.
A "step" is one environment step of all environments of a rank.

Own arm, printed as ONE JSON line by rank 0:
  value     env-steps/sec, whole job, actions resident in HBM ([T, N] int8),
            observations written to a [T, N, 147] rollout buffer (385 MB > L2).
            The timed region is ALWAYS calls of bb_pool_rollout (the persistent
            stepping kernel, T = 40 steps per launch) covering exactly K steps:
            K // T whole rollouts and one of K % T steps; CUDA events, barrier +
            synchronize on both sides, max over ranks.
  roofline  achieved = 153 algorithmic bytes per env-step (147 obs + 4 reward +
            1 done + 1 action; SURVEY.md 8d) x the per-GPU `value` of that SAME
            timed region, against MEASURED_PEAKS.json hbm_gbs; `kernel_frac` is
            the same figure for the stepping kernel alone (CUDA events around it,
            bb_pool_rollout_timed).
  e2e       the same metric through the reference-facing C-ABI host-buffer call
            (bb_pool_step_host = what ParallelEnv.step hands BaseAlgo): actions
            host->device and obs/reward/done/direction device->host inside the
            timed region, every step, >= 200 steps; per-rank min/median/max.
  facade_e2e  the reference-SHAPED Python facade (vecenv.ParallelEnv.step: N obs
            dicts per step) -- host bound by construction, a few steps only.
  cpu_baseline  the oracle's C port of the same path on this box's host cores.
  reference_parallel_env  the reference's own ParallelEnv (64 procs) when a
            reference tree is reachable (build container), else available: false.

--impl reference: the CPU arm (oracle C port, all host threads, same workload);
the reference itself is Python on a third-party package that is absent here
and /root/reference does not exist on the GPU box (see DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVEL = 'GoToLocal'
N_ENVS = 65536
CHUNK = int(os.environ.get("BENCH_CHUNK", "40"))   # rollout length per launch (= --frames-per-proc, arguments.py:42)
MIN_HOST_STEPS = 200            # ... and the per-step legs (e2e, per_step_api) never fewer than this
ALGO_BYTES_PER_STEP = 153       # 147 obs + 4 reward + 1 done + 1 action (SURVEY.md 8d)
FALLBACK_HBM_GBS = 6650.0       # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = 'env-steps/sec at 65 536 envs (GoToLocal); obs bit-exact vs CPU ref'


def workload(level, n):
    """config.workload -- the SAME string in both arms"""
    return 'BabyAI-%s-v0, %d envs/GPU, uniform random actions, ParallelEnv auto-reset, in-kernel verifier' % (level, n)


def hbm_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured'
        except Exception:
            pass
    return FALLBACK_HBM_GBS, 'fallback'


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[2 + k].lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def cpu_port(level, steps_budget_s, n_envs, threads):
    """Oracle C port (oracle/babyai_oracle.c) on the host cores: random actions, auto-reset."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import oracle as orc
    pool = orc.OraclePool(level, n_envs, np.array([100 + i for i in range(n_envs)], dtype=np.uint64))
    pool.reset()
    rng = np.random.RandomState(0)
    acts = rng.randint(0, 7, (64, n_envs)).astype(np.int8)
    for k in range(2):
        pool.step(acts[k], nthreads=threads)
    t0 = time.perf_counter()
    k = 0
    while True:
        pool.step(acts[k % 64], nthreads=threads)
        k += 1
        if time.perf_counter() - t0 > steps_budget_s:
            break
    dt = time.perf_counter() - t0
    return n_envs * k / dt, k


def reference_parallel_env(level, procs=64, steps=300):
    """north_star's side-by-side number: the reference's OWN ParallelEnv (penv.py:4-59, one forked process per env) over
    envs built as scripts/train_rl.py:53-60 does, timed around ParallelEnv.step -- possible only where a reference tree is
    reachable (BABYAI_REFERENCE or /root/reference: the build container).  The GPU box has none: say so."""
    ref = os.environ.get('BABYAI_REFERENCE', '/root/reference')
    if os.environ.get('BENCH_REF_PENV', '1') == '0':
        return {'available': False, 'why': 'disabled (BENCH_REF_PENV=0)'}
    if not os.path.isdir(os.path.join(ref, 'babyai', 'levels')):
        return {'available': False, 'why': 'no reference tree at %s (the GPU box has none); measured in the build container: '
                                           'see DESIGN.md section 7 / profiles/r02_reference_parallel_env.json' % ref}
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'oracle', 'bench_ref_parallel_env.py'), '--level', level,
                            '--procs', str(procs), '--steps', str(steps), '--warmup', '30'],
                           capture_output=True, text=True, timeout=600)
        lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
        if not lines:
            return {'available': False, 'why': (r.stderr or 'no output')[-300:]}
        d = json.loads(lines[-1])
        d['available'] = True
        d['value'] = d['parallel_env_steps_per_s']
        d['unit'] = 'env-steps/s'
        return d
    except Exception as ex:
        return {'available': False, 'why': repr(ex)[:300]}


def run_reference(args, rank):
    """CPU arm: the oracle port with every host thread, same workload and metric."""
    if rank != 0:
        return
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import oracle as orc
    threads = os.cpu_count() or 1
    n = args.envs
    pool = orc.OraclePool(args.level, n, np.array([100 + i for i in range(n)], dtype=np.uint64))
    pool.reset()
    acts = np.random.RandomState(0).randint(0, 7, (64, n)).astype(np.int8)
    t0 = time.perf_counter()
    pool.step(acts[0], nthreads=threads)
    per_step = time.perf_counter() - t0
    # keep the whole run within ~2 minutes: if needed a step covers only the first `m` environments
    total = per_step * (args.steps + args.warmup)
    m = n
    if total > 120:
        m = max(1024, int(n * 120 / total) // 1024 * 1024)
        pool = orc.OraclePool(args.level, m, np.array([100 + i for i in range(m)], dtype=np.uint64))
        pool.reset()
        acts = acts[:, :m].copy()
    for k in range(args.warmup):
        pool.step(acts[k % 64], nthreads=threads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        pool.step(acts[k % 64], nthreads=threads)
    dt = time.perf_counter() - t0
    v = m * args.steps / dt
    sample = '%d steps x %d envs (of %d) of %s, oracle C port, %d host threads' % (args.steps, m, n, args.level, threads)
    out = {
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'env-steps/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps * (n / m),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
        'config': {'workload': workload(args.level, n), 'envs_per_step_sampled': m,
                   'execution': 'oracle/babyai_oracle.c (C restatement of the reference path), %d host threads' % threads},
        'cpu_baseline': {'value': v, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'reference_parallel_env': reference_parallel_env(args.level),
    }
    print(json.dumps(out), flush=True)


def write_outputs(out_dir, arrays, limit=64 << 20):
    """arrays: name -> float32 array whose first axis is the environment.  Writes out_dir/<name>.npy; when all of them
    together exceed `limit` bytes, only a fixed, seeded sample of environments (listed in env_index.npy)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = len(arrays['reward'])
    per_env = sum(a.nbytes for a in arrays.values()) // n
    if n * per_env > limit:
        idx = np.sort(np.random.RandomState(0).choice(n, (limit - 4096) // (per_env + 8), replace=False))
        arrays = dict({k: a[idx] for k, a in arrays.items()}, env_index=idx.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=200)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--envs', type=int, default=N_ENVS, help='environments per GPU')
    ap.add_argument('--level', default=LEVEL)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--brief', action='store_true', help='device-resident value + kernel timing only (child runs of --other-configs)')
    ap.add_argument('--lean', action='store_true', help='value, roofline and e2e only (multi-GPU scaling runs of the other configs)')
    ap.add_argument('--no-other-configs', action='store_true', help='skip the child runs of BASELINE configs 3-5 (per-GPU share)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step returned to rank 0 (obs, reward, done, '
                                                          'direction) as DIR/<name>.npy, float32')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference(args, rank)
        return

    # one rank per GPU: bind the rank to its GPU's NUMA node before the CUDA context and any page-locked buffer exist
    from babyai_b200.sharding import gather_counters, pin_to_gpu_numa, shard_seeds
    numa = pin_to_gpu_numa(local_rank) if os.environ.get('BENCH_NO_NUMA_PIN') is None else None

    import numpy as np
    import torch
    import torch.distributed as dist
    from babyai_b200 import BabyAIVecEnv

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the pool has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_f64(x):
        """per-rank float -> list over ranks (all-gather of one double)"""
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world == 1:
            return [float(x)]
        parts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        return [float(p.item()) for p in parts]

    n, K, W = args.envs, args.steps, args.warmup
    T = CHUNK
    # rank r owns global env indices [r*n, (r+1)*n); seeds follow the global index (train_rl.py:59, --seed 1)
    seeds = shard_seeds(1, world * n, rank, world)
    env = BabyAIVecEnv(args.level, n, seeds=seeds, device=local_rank)
    env.reset()

    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = torch.randint(0, 7, (T, n), device=dev, dtype=torch.int8, generator=gen)
    obs = torch.empty((T, n, 7, 7, 3), dtype=torch.uint8, device=dev)       # 385 MB at n = 65 536: larger than L2
    rew = torch.empty((T, n), dtype=torch.float32, device=dev)
    done = torch.empty((T, n), dtype=torch.uint8, device=dev)
    dirs = torch.empty((T, n), dtype=torch.int8, device=dev)

    bufs = (actions, obs, rew, done, dirs)

    def run_rollouts(r, bufs=bufs):
        for _ in range(r):
            env.rollout(*bufs)

    # ---- device-resident throughput: exactly K steps, K // T whole rollouts and one of K % T steps ----
    n_roll, K_rest = divmod(K, T)
    rest_bufs = [b[:K_rest] for b in bufs]
    w_roll = max((max(W, 3) + T - 1) // T, 2)
    run_rollouts(w_roll)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = env.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    run_rollouts(n_roll)
    if K_rest:
        run_rollouts(1, rest_bufs)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = env.launches() - l0
    if args.dump_outputs and rank == 0:
        last = (K_rest or T) - 1
        dump = {'obs': obs[last], 'reward': rew[last], 'done': done[last], 'direction': dirs[last]}
        dump = {k: v.cpu().numpy().astype(np.float32) for k, v in dump.items()}
    # keep the GPU busy a little longer so the clock sampler sees load even for short K
    clocks = None
    if rank == 0:
        t_end = time.time() + 0.4
        while time.time() < t_end:
            run_rollouts(4)
            torch.cuda.synchronize()
        clocks = sampler.stop()
    ms_ranks = gather_f64(ms)
    ms = max(ms_ranks)

    # ---- per-kernel timing: the stepping kernel of one rollout launch, CUDA events on its stream ----
    kr, kf = [], []
    for t in range(16):
        a, b = env.rollout_timed(actions, obs, rew, done, dirs)
        if t >= 4 and a > 0:
            kr.append(a); kf.append(b)          # b = 0 for the launches that do not refill
    k_roll_ms = sum(kr) / len(kr) if kr else 0.0
    k_refill_ms = sum(kf) / len(kf) if kf else 0.0      # amortised per launch

    peak, peak_src = hbm_peak()
    value = world * n * K / (ms * 1e-3)
    achieved = ALGO_BYTES_PER_STEP * (value / world) / 1e9           # GB/s of algorithmic bytes per GPU, SAME timed region
    kernel_achieved = ALGO_BYTES_PER_STEP * n * T / (k_roll_ms * 1e-3) / 1e9 if k_roll_ms > 0 else 0.0
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, dump)
    if args.brief:
        if rank == 0:
            print(json.dumps({'level': args.level, 'envs_per_gpu': n, 'value': value, 'us_per_step': 1e3 * ms / K, 'steps': K,
                              'kernel_us_per_step': 1e3 * k_roll_ms / T, 'refill_ms_per_launch': k_refill_ms,
                              'roofline_frac': achieved / peak, 'counters': env.counters()}), flush=True)
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- the per-step entry point (policy in the loop): bb_pool_step on device buffers, one launch per step ----
    Ks = max(min(K, 600), MIN_HOST_STEPS) if not args.lean else 40
    for t in range(20):
        env.step(actions[t % T], obs[t % T], rew[t % T], done[t % T], dirs[t % T])
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for t in range(Ks):
        env.step(actions[t % T], obs[t % T], rew[t % T], done[t % T], dirs[t % T])
    s1.record()
    barrier()
    per_step_ms = max(gather_f64(s0.elapsed_time(s1) / Ks))

    # ---- end to end through the host-buffer C-ABI call --------------------------------------------
    h_act = np.random.RandomState(7 + rank).randint(0, 7, (64, n)).astype(np.int8)
    # page-locked host buffers (what babyai_b200.ParallelEnv hands to bb_pool_step_host)
    pins = [torch.zeros((n, 7, 7, 3), dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.float32).pin_memory(),
            torch.zeros(n, dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.int8).pin_memory()]
    h_obs, h_rew, h_done, h_dir = [t.numpy() for t in pins]
    Ke = max(min(K, 400), MIN_HOST_STEPS)
    for k in range(10):
        env.step_host(h_act[k], h_obs, h_rew, h_done, h_dir)
    barrier()
    t0 = time.perf_counter()
    for k in range(Ke):
        env.step_host(h_act[k % 64], h_obs, h_rew, h_done, h_dir)
    own_s = time.perf_counter() - t0             # this rank's own loop (bb_pool_step_host synchronises its stream)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_ranks = sorted(n * Ke / s for s in gather_f64(own_s))
    e2e_s = max(gather_f64(e2e_s))

    # ---- RGB partial observations (RGBImgPartialObsWrapper, the 'pixel' architectures' input): the one HBM-bound output ----
    # obs uint8[N,7,7,3] -> uint8[N,56,56,3]: 9 408 B written per 147 B read; 616 MB per call at N = 65 536 (> L2)
    rgb = {}
    try:
        if args.lean:
            raise RuntimeError('skipped (--lean)')
        pics = torch.empty((n, 56, 56, 3), dtype=torch.uint8, device=dev)
        for k in range(3):
            env.render_rgb(obs[k % T], pics)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        r0.record()
        for k in range(reps):
            env.render_rgb(obs[k % T], pics)
        r1.record()
        torch.cuda.synchronize()
        rms = r0.elapsed_time(r1) / reps
        rbytes = n * (56 * 56 * 3 + 147)
        rgb = {'kernel': 'k_render_rgb', 'ms': rms, 'algorithmic_bytes': rbytes, 'achieved': rbytes / (rms * 1e-3) / 1e9, 'unit': 'GB/s',
               'frac': rbytes / (rms * 1e-3) / 1e9 / peak, 'bound': 'hbm', 'frames_per_s': n / (rms * 1e-3),
               'api': 'bb_pool_render_rgb: obs uint8[N,7,7,3] -> uint8[N,56,56,3] (tile size 8), device buffers'}
        del pics
    except Exception as ex:
        rgb = {'error': repr(ex)[:300]}

    # ---- the only collective on this path: all-gather of the counters --------------------
    cnt = gather_counters(env.counters(), device=dev)

    # ---- the learner-facing path with observations resident in HBM (babyai_b200.learner; informational) ----------
    # per step: actions host->device, the step kernel writing into a fresh observation tensor, ObssPreprocessor handing
    # the model image float[N,7,7,3] + instr long[N,L] on the device, reward/done device->host.  Measured on this rank.
    learner = {}
    for key, fused_io in ((('fused_io', True), ('tensor_copies', False)) if not args.lean else ()):
        # fused_io (default): bb_pool_step_learner (actions / reward / done over mapped page-locked memory inside the step call);
        # tensor_copies: bb_pool_step + torch copies of those three
        try:
            from babyai_b200 import make_envs
            from babyai_b200.learner import DeviceParallelEnv, ObssPreprocessor
            denv = DeviceParallelEnv(make_envs(args.level, n), pool=env, fused_io=fused_io)
            pre = ObssPreprocessor(trim=False)
            ob = denv.reset()
            Kl = max(min(K, 300), MIN_HOST_STEPS)
            for k in range(5):
                pre(ob, device=dev)
                ob, _r, _d, _i = denv.step(h_act[k])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(Kl):
                pre(ob, device=dev)
                ob, _r, _d, _i = denv.step(h_act[k % 64])
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            learner[key] = {'value_per_gpu': n * Kl / dt, 'unit': 'env-steps/s', 'steps': Kl, 'h2d_bytes_per_step': n,
                            'd2h_bytes_per_step': n * 5}
        except Exception as ex:          # informational leg: never lose the bench line over it
            learner[key] = {'error': repr(ex)[:300]}
    learner['api'] = 'DeviceParallelEnv.step + ObssPreprocessor (observations stay in HBM); fused_io is the default'

    # ---- the reference-SHAPED facade: vecenv.ParallelEnv.step builds N Python obs dicts per step (rank 0, single-GPU runs) ----
    facade = None
    if rank == 0 and world == 1 and not args.lean:
        try:
            from babyai_b200 import ParallelEnv, make_envs
            nf = min(n, 4096)                     # penv-sized: the dict facade is host bound by orders of magnitude
            pe = ParallelEnv(make_envs(args.level, nf))
            pe.reset()
            fa = np.random.RandomState(3).randint(0, 7, (8, nf))
            for k in range(2):
                list(pe.step(fa[k]))
            t0 = time.perf_counter()
            for k in range(2, 8):
                list(pe.step(fa[k]))
            dt = time.perf_counter() - t0
            facade = {'value': nf * 6 / dt, 'unit': 'env-steps/s', 'envs': nf, 'steps': 6,
                      'api': 'babyai_b200.ParallelEnv.step (penv.py surface: tuple of N obs dicts, rewards, dones, infos); '
                             'host bound: the per-env Python objects dominate'}
            pe.pool.close()
        except Exception as ex:
            facade = {'error': repr(ex)[:300]}

    # ---- BASELINE configs 3-5 at their per-GPU size, each in a child process (single-GPU default runs only) ----
    others = None
    if rank == 0 and world == 1 and not args.no_other_configs and args.level == LEVEL and n == N_ENVS:
        others = {}
        # steady state: a fresh pool starts all its episodes at once, so on the multi-room levels (episodes of 576 .. 4 608
        # steps) hardly any level is consumed -- and generated -- during the first thousand steps: a 1 000-step run read 5.2e9 /
        # 4.9e9 on GoTo / BossLevel where 200 000 steps give 4.5e9 / 4.4e9 (r02m vs r02r).  The warm-up runs past the longest
        # time-out and the timed region covers several thousand episodes per env slot.
        for key, lv, ne, ks, kw in (('C3 PickupLoc', 'PickupLoc', 65536, 4000, 400), ('C4 GoTo', 'GoTo', 32768, 40000, 6000),
                                    ('C5 BossLevel (per-GPU share)', 'BossLevel', 32768, 40000, 6000)):
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), '--brief', '--level', lv, '--envs', str(ne),
                                    '--steps', str(ks), '--warmup', str(kw)], capture_output=True, text=True, timeout=150)
                lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
                others[key] = json.loads(lines[-1]) if lines else {'error': (r.stderr or 'no output')[-400:], 'returncode': r.returncode}
            except subprocess.TimeoutExpired:
                others[key] = {'error': 'timed out after 150 s (child killed); remaining configs skipped'}
                break
            except Exception as ex:
                others[key] = {'error': repr(ex)[:300]}

    if rank == 0:
        traffic = None
        tp = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get('k_rollout_dram_bytes_per_launch')
            except Exception:
                traffic = None
        out = {
            'metric': METRIC, 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'steps_requested': K,
            'warmup': w_roll * T, 'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'u8', 'data': 'synthetic',
            'config': {'workload': workload(args.level, n),
                       'envs_per_gpu': n, 'rollout_chunk': T,
                       'l2_policy': 'obs written to a [%d, %d, 147] buffer (%.0f MB) larger than L2' % (T, n, T * n * 147 / 1e6),
                       'execution': 'timed region = %d calls of bb_pool_rollout (%d steps each) and %d of %d steps: one persistent '
                                    'stepping kernel per call with the env state resident in shared memory; level generation inside it '
                                    '(single-room levels) or beside it on a side stream' % (n_roll, T, 1 if K_rest else 0, K_rest),
                       'actions': 'int8 [T, N], resident in HBM',
                       'parallelism': 'replicas x%d, counters all-gather only' % world,
                       'numa': numa},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': traffic, 'kernel': 'k_rollout', 'from': 'value / n_gpus x 153 B (the timed region above)',
                         'kernel_achieved': kernel_achieved, 'kernel_frac': kernel_achieved / peak,
                         'kernel_ms': k_roll_ms, 'steps_per_launch': T,
                         'kernel_us_per_step': 1e3 * k_roll_ms / T, 'refill_ms_per_launch': k_refill_ms,
                         'algorithmic_bytes_per_launch': ALGO_BYTES_PER_STEP * n * T, 'peak_source': peak_src},
            'per_step_api': {'value': world * n / (per_step_ms * 1e-3), 'unit': 'env-steps/s', 'ms_per_step': per_step_ms,
                             'api': 'bb_pool_step (one launch per step; level generation on a side stream), device buffers', 'steps': Ks},
            'e2e': {'value': world * n * Ke / e2e_s, 'unit': 'env-steps/s', 'h2d_bytes_per_step': n,
                    'd2h_bytes_per_step': n * (147 + 4 + 1 + 1), 'steps': Ke,
                    'api': 'bb_pool_step_host (the C-ABI call, not the Python dict facade), page-locked host buffers',
                    'per_rank': {'min': e2e_ranks[0], 'median': e2e_ranks[len(e2e_ranks) // 2], 'max': e2e_ranks[-1]}},
            'rgb_roofline': rgb,
            'facade_e2e': facade,
            'learner_path': learner,
            'other_configs': others,
            'reference_parallel_env': reference_parallel_env(args.level),
            'gpu_launches': int(launches),
            'ms_per_rank': ms_ranks,
            'clocks': clocks,
            'counters': cnt,
        }
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            v, k = cpu_port(args.level, 12.0, n, threads)
            out['cpu_baseline'] = {'value': v, 'unit': 'env-steps/s', 'cores': threads, 'kind': 'port',
                                   'sample': '%d steps x %d envs of %s, oracle C port, %d host threads' % (k, n, args.level, threads)}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
