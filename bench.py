#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched Crazyflie stepping engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA engine
    python bench.py --impl reference [--gpus N] --steps K ...    # CPU arm (oracle port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...        # one rank per GPU

Workload (BASELINE.json configs[1], SURVEY.md 8d "Config 2"): DroneHoverSimpleEnv-v0,
65,536 lock-step environments per GPU, 10 % domain randomisation, observation noise on,
history H = 2, float32 SoA state, on-device Philox, U(-1,1) float32 actions, auto-reset.

One bench "step" = `--launches` (default 16) rollout segments of `--inner` (default 64) env.steps
of every environment = 1,024 env.steps per environment, each segment ONE fused launch writing
into [inner, N, .] rollout tensors.  Actions and observations stream through ring buffers larger
than L2; the 65,536-env state itself (~13 MB) is L2-resident by the workload's definition --
`config.l2` says so, and `roofline_hbm_resident_off` repeats the measurement at 4 Mi environments
per GPU where the state (0.9 GB) cannot stay in L2.  Multi-GPU: the episode statistics of a bench
step are combined across ranks ONCE per step (the reference reduces them once per epoch,
utils/loggers.py:519-524) with an asynchronous NCCL all-gather that overlaps the next step.

JSON keys follow the driver contract: value (device-resident inputs, CUDA events, max over
ranks), e2e (host buffers, H2D/D2H inside the timed region), roofline, cpu_baseline, clocks,
gpu_launches.  Only the `cpu_baseline` leg and `--impl reference` execute oracle/.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENV_ID = 'DroneHoverSimpleEnv-v0'
METRIC = 'env-steps/sec'
UNIT = 'env-steps/s'
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 60 * 1000 * 1000    # --dump-outputs: upper bound of the arrays written
HBM_FALLBACK_GBS = 6650.0        # /opt/skills/guides/B200_PROFILING.md fallback


# =============================================================================================
#  CPU arm: the oracle port (numpy restatement of the reference env), one env per process --
#  the reference's own parallel model is one env per MPI rank (algs/iwpg/iwpg.py:90).
# =============================================================================================
def _cpu_worker(args):
    env_id, seed, budget_s, max_steps = args
    import numpy as np
    from oracle.phoenix_oracle import OracleEnv, NumpyGlobalSource
    np.random.seed(seed)
    env = OracleEnv(env_id, NumpyGlobalSource())
    rng = np.random.default_rng(seed)
    env.reset()
    acts = rng.uniform(-1, 1, (4096, 4)).astype(np.float32)
    n, ep_len = 0, 0
    t0 = time.perf_counter()
    while True:
        _, _, terminated, _, _ = env.step(acts[n & 4095])
        n += 1
        ep_len += 1
        if terminated or ep_len == 500:
            env.reset()
            ep_len = 0
        if (n & 63) == 0 and time.perf_counter() - t0 >= budget_s:
            break
        if max_steps and n >= max_steps:
            break
    return n, time.perf_counter() - t0


def cpu_env_steps_per_sec(env_id, budget_s, procs=None, max_steps=0, pool=None):
    """Σ steps / wall over `procs` worker processes (default: all host cores)."""
    import multiprocessing as mp
    procs = procs or os.cpu_count() or 1
    own = pool is None
    if own:
        pool = mp.get_context('fork').Pool(procs)
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, [(env_id, 1000 + 10000 * r, budget_s, max_steps) for r in range(procs)], chunksize=1)
    wall = time.perf_counter() - t0
    if own:
        pool.close()
        pool.join()
    steps = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return steps / busy, procs, steps, wall


def run_reference_arm(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    K, W = a.steps, a.warmup
    per_step_budget = min(2.0, 120.0 / max(1, K + W))          # whole run ends within minutes
    procs = os.cpu_count() or 1
    pool = mp.get_context('fork').Pool(procs)
    for _ in range(W):
        cpu_env_steps_per_sec(a.env_id, per_step_budget / 4, procs, pool=pool)
    tot_steps, tot_time = 0, 0.0
    for _ in range(K):
        v, _, steps, _ = cpu_env_steps_per_sec(a.env_id, per_step_budget, procs, pool=pool)
        tot_steps += steps
        tot_time += steps / v
    pool.close()
    pool.join()
    value = tot_steps / tot_time
    sample = (f'{K} samples of {per_step_budget:.2f} s on {procs} processes, one oracle env per process, '
              f'U(-1,1) float32 actions, auto-reset ({tot_steps} env-steps in total)')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': K,
        'warmup': W, 'ms_per_step': 1e3 * tot_time / K, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(a, a.num_envs),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': procs, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# =============================================================================================
#  clocks during the timed region (NVML; same fields as the recipe's nvidia-smi line)
# =============================================================================================
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.thread = None

    def _reasons(self, mask):
        nv = self.nv
        names = {'hw_slowdown': 'nvmlClocksThrottleReasonHwSlowdown',
                 'hw_thermal_slowdown': 'nvmlClocksThrottleReasonHwThermalSlowdown',
                 'sw_thermal_slowdown': 'nvmlClocksThrottleReasonSwThermalSlowdown',
                 'sw_power_cap': 'nvmlClocksThrottleReasonSwPowerCap',
                 'hw_power_brake': 'nvmlClocksThrottleReasonHwPowerBrakeSlowdown'}
        return {k for k, attr in names.items() if mask & getattr(nv, attr, 0)}

    def sample_once(self):
        nv = self.nv
        if nv is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.reasons |= self._reasons(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        except Exception:
            pass

    def _loop(self):
        while not self.stop_flag:
            self.sample_once()
            time.sleep(0.001)

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def halt(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join()
            self.thread = None

    def stop(self):
        self.halt()
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(s)}


def workload_config(a, n_per_gpu):
    return {'workload': f'{a.env_id}, {n_per_gpu} lock-step envs per GPU, DR 0.10, observation noise on, '
                        f'H=2, U(-1,1) actions, auto-reset (BASELINE.json configs[1])',
            'env_id': a.env_id, 'envs_per_gpu': n_per_gpu, 'env_steps_per_bench_step': a.launches * a.inner * n_per_gpu,
            'inner_env_steps': a.inner, 'launches_per_bench_step': a.launches, 'launch': a.mode,
            'rng': 'philox4x32-10 on device',
            'l2': 'actions and observations stream through ring buffers larger than L2; the per-env state '
                  'is L2-resident at this size by the workload definition (see roofline_hbm_resident_off)'}


# =============================================================================================
#  GPU arm
# =============================================================================================
class Segment:
    """One rollout segment: `inner` env.steps into [inner, N, .] tensors of a ring of segments.
    mode 'fused': one pdx_step_many launch per segment; 'per-step': `inner` pdx_step launches."""

    def __init__(self, env, inner, n_ring, gen, mode='fused', near_hover=False):
        import torch
        n, d, dev = env.num_envs, env.obs_dim, env.device
        self.env, self.inner, self.n_ring, self.mode = env, inner, n_ring, mode
        if near_hover:        # SURVEY 8d "fixed policy": a = HOVER_ACTION + N(0, 0.05), ~2 % of envs finish per step
            self.actions = env.cfg.hover_action + 0.05 * torch.randn((n_ring, inner, n, 4), device=dev, generator=gen)
        else:                 # U(-1, 1): ~11 % of envs finish per step
            self.actions = torch.rand((n_ring, inner, n, 4), device=dev, generator=gen) * 2 - 1
        self.obs = torch.empty((n_ring, inner, n, d), dtype=env.dtype, device=dev)
        self.reward = torch.empty((n_ring, inner, n), dtype=env.dtype, device=dev)
        self.cost = torch.empty((n_ring, inner, n), dtype=env.dtype, device=dev)
        self.terminated = torch.empty((n_ring, inner, n), dtype=torch.uint8, device=dev)
        self.truncated = torch.empty((n_ring, inner, n), dtype=torch.uint8, device=dev)
        self.seg_outs = [{'obs': self.obs[r], 'reward': self.reward[r], 'cost': self.cost[r],
                          'terminated': self.terminated[r], 'truncated': self.truncated[r]} for r in range(n_ring)]
        self.outs = [[{k: v[t] for k, v in self.seg_outs[r].items()} for t in range(inner)] for r in range(n_ring)]

    def run(self, k):
        r = k % self.n_ring
        env = self.env
        if self.mode == 'fused':
            env.step_many(self.actions[r], self.seg_outs[r])
            return 1
        acts, outs = self.actions[r], self.outs[r]
        for t in range(self.inner):
            env.step(acts[t], out=outs[t])
        return self.inner


def ring_slots(bytes_per_segment):
    return max(2, -(-2 * L2_BYTES // bytes_per_segment))


def dump_outputs(seg, k, out_dir, max_bytes=DUMP_BYTES):
    """Writes what segment `k` returned to its caller (obs [inner, S, D], reward / cost / terminated / truncated
    [inner, S]) as out_dir/<name>.npy in float32, for a fixed, seeded sample of S environments (S as large as
    `max_bytes` allows, all of them when they fit), so that two builds can be compared output for output."""
    import numpy as np
    import torch
    outs = seg.seg_outs[k % seg.n_ring]
    inner, n, d = outs['obs'].shape
    s = min(n, max(1, max_bytes // (inner * (d + 4) * 4)))
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:s].sort().values.to(outs['obs'].device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outs.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.index_select(1, idx).float().cpu().numpy())


def time_device(env, seg, K, W, dist_ctx, sampler=None, per_step=1):
    """K bench steps of `per_step` segments each, timed with CUDA events on the launching stream; max
    over ranks.  `sampler`: clocks are read ONLY between the two events (the sampler thread is started
    after the first and this thread keeps sampling until the second has completed)."""
    import torch
    launches = 0
    for k in range(W * per_step):
        seg.run(k)
        if (k + 1) % per_step == 0:
            dist_ctx.reduce_stats(env)
    dist_ctx.flush_stats()
    dist_ctx.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if sampler is not None:
        sampler.start()
    for k in range(K * per_step):
        launches += seg.run(W * per_step + k)
        if (k + 1) % per_step == 0:
            dist_ctx.reduce_stats(env)
    dist_ctx.flush_stats()
    e1.record()
    if sampler is not None:
        while not e1.query():
            time.sleep(0.0005)
        sampler.halt()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    dist_ctx.barrier()
    return dist_ctx.max_over_ranks(ms), launches


def time_e2e(env, inner, K, W, dist_ctx, gen_seed):
    """Same metric through the public VecEnv API with HOST buffers (VecEnv.step_many_host): every
    segment copies its actions from pinned host memory, runs, and copies obs / reward / cost /
    flags back to pinned host memory, chunk-pipelined over three streams; all inside the timed
    region."""
    import torch
    chunk = 8 if inner % 8 == 0 else 1
    pipe = env.make_host_pipeline(inner, chunk)
    g = torch.Generator().manual_seed(gen_seed)
    pipe['host']['actions'].copy_(torch.rand(pipe['host']['actions'].shape, generator=g) * 2 - 1)
    for _ in range(W):
        env.step_many_host(pipe)
    dist_ctx.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        env.step_many_host(pipe)
    e1.record()
    torch.cuda.synchronize()
    ms = dist_ctx.max_over_ranks(e0.elapsed_time(e1))
    dist_ctx.barrier()
    assert torch.isfinite(pipe['host']['obs']).all()
    return ms, pipe['h2d_bytes'], pipe['d2h_bytes']


def link_ceiling(dev, dist_ctx, mbytes=512, reps=4):
    """What this box's host link gives a rank while ALL ranks copy at the same time: pinned D2H alone, and D2H with a
    concurrent H2D of 1/9 of the size (the e2e leg's ratio), GB/s per rank -- the ceiling the e2e number is a
    fraction of (its timed region moves d2h_bytes_per_step over this link)."""
    import torch
    n = mbytes << 20
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    d2 = torch.empty(n // 9, dtype=torch.uint8, device=dev)
    h2 = torch.empty(n // 9, dtype=torch.uint8).pin_memory()
    s_out, s_in = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    out = {}
    for both in (False, True):
        for timed in (False, True):
            dist_ctx.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s_out)
            for _ in range(reps if timed else 1):
                with torch.cuda.stream(s_out):
                    h.copy_(d, non_blocking=True)
                if both:
                    with torch.cuda.stream(s_in):
                        d2.copy_(h2, non_blocking=True)
            e1.record(s_out)
            torch.cuda.synchronize()
            ms = dist_ctx.max_over_ranks(e0.elapsed_time(e1))
        out['d2h_with_h2d_gbs' if both else 'd2h_gbs'] = reps * n / (ms * 1e-3) / 1e9
    return out


def bind_to_gpu_numa_node(local_rank):
    """Host side of the e2e leg: keep this rank's threads (and therefore its pinned staging buffers,
    first-touch) on the NUMA node its GPU hangs off; otherwise eight ranks share one node's memory
    controllers.  Best effort: silently skipped where sysfs does not tell."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = f'{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0'
        with open(f'/sys/bus/pci/devices/{bdf}/numa_node') as f:
            node = int(f.read())
        if node < 0:
            return None
        with open(f'/sys/devices/system/node/node{node}/cpulist') as f:
            cpus = set()
            for part in f.read().strip().split(','):
                lo, _, hi = part.partition('-')
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def ppo_rollout_leg(dev, n=131072, T=64, rollouts=4):
    """BASELINE.json configs[4] next to the headline: DroneHoverBulletEnv-v0 driving a PPO rollout on this GPU:
    IWPGAlgorithm.roll_out's loop in ONE persistent kernel per rollout (pdx_collect: policy networks on the
    tcgen05 tensor cores between two env.steps of a thread, environment state in registers), then GAE and the
    running statistics, all on device.  Reported per operand precision of the policy networks and, for
    comparison, for the two-kernel path (policy kernel and env.step kernel alternating);
    bench_configs.py measures the same under torchrun."""
    import torch
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector

    def run(kernel, fused):
        torch.manual_seed(0)
        env = VecEnv('DroneHoverBulletEnv-v0', n, device=dev, seed=2, keep_final_obs=True)
        ac = ActorCritic(env.obs_dim, device=dev, policy_kernel=kernel)
        col = RolloutCollector(env, ac, T)
        col.use_fused_kernel = fused
        for _ in range(3):              # the first programmatic-dependent launches of a process carry a one-time cost
            col.update_running_statistics(col.collect())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(rollouts):
            data = col.collect()
            col.update_running_statistics(data)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        assert col.fused_used == fused
        return {'value': rollouts * T * n / (ms * 1e-3), 'unit': UNIT, 'ms_per_rollout': ms / rollouts,
                'gpu_launches_per_rollout': (1 if fused else 2 * T) + 8}

    out = {'workload': f'DroneHoverBulletEnv-v0, {n} envs x {T} steps per rollout, reference PPO networks (pi 50-50 relu, '
                       'v 64-64 tanh): policy step + env.step + GAE + running statistics (BASELINE.json configs[4])'}
    names = {'tc': 'split TF32 (float32-level results)', 'tc_tf32': 'single TF32 (1e-3 relative on mu / v)'}
    for kernel in ('tc', 'tc_tf32'):
        out[f'pdx_collect, {names[kernel]}'] = run(kernel, True)
    out[f'k_policy_tc + k_rollout alternating, {names["tc_tf32"]}'] = run('tc_tf32', False)
    best = max((v for v in out.values() if isinstance(v, dict)), key=lambda r: r['value'])
    out['value'], out['unit'] = best['value'], UNIT
    return out


class DistCtx:
    def __init__(self, n_gpus):
        import torch
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(self.local_rank)
        self.numa_node = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        self.device = torch.device('cuda', self.local_rank)
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            # The caller's NCCL_DEBUG is left alone (the driver reads NCCL's rank / topology lines).  stdout
            # carries ONE JSON line, so NCCL's log goes to stderr unless the caller chose a file.
            if os.environ.get('NCCL_DEBUG') and not os.environ.get('NCCL_DEBUG_FILE'):
                os.environ['NCCL_DEBUG_FILE'] = '/dev/stderr'
            # NCCL prints its version banner with printf on fd 1 whatever NCCL_DEBUG_FILE says: fd 1 points at
            # stderr while the communicator comes up (init + first collective), then stdout is restored
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group('nccl', device_id=self.device)
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
            self.dist = dist
        else:
            self.dist = None
        import torch as _t
        self.episodes = _t.zeros((), dtype=_t.float64, device=self.device)   # finished episodes, all ranks
        self._pending = None

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def max_over_ranks(self, x):
        if not self.dist:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_stats(self, env):
        """Episode-return statistics across ranks: the only cross-GPU traffic of the path, once per
        bench step (SURVEY.md 8e; replaces utils/mpi_tools.py:217-240, which the reference runs once per
        epoch, utils/loggers.py:519-524).  The all-gather is asynchronous (NCCL's own stream); its result
        is combined one step later, so the collective never sits between two env.step launches."""
        if not self.dist:
            return
        from phoenix_drone_simulation_b200.rollout import gather_episode_stats_async
        self.flush_stats()
        # this step's statistics only (the collector's flow: roll out, combine, log, clear)
        self._pending = gather_episode_stats_async(env.episode_stats(clear=True), self.dist)

    def flush_stats(self):
        if self._pending is not None:
            self.episodes.add_(self._pending()[0])
            self._pending = None

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def kernel_source_hash():
    """sha256 over the sources the step kernel is compiled from: ties profile counters to a build."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, 'phoenix_drone_simulation_b200', 'csrc')
    for f in ('pdx_kernels.cuh', 'pdx_model.cuh', 'pdx_math.cuh', 'pdx_layout.h', 'pdx_dispatch.cuh'):
        with open(os.path.join(csrc, f), 'rb') as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def profile_counters(env_steps_per_launch):
    """Per-launch ncu counters of the bench's step kernel (profiles/rollout_counters.json, written by
    profiles/export_summary.py from an `ncu --set full` capture of this command).  `stale` = the kernel
    sources changed since the capture (the counts then describe an older build)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'rollout_counters.json')) as f:
            c = json.load(f)
        if c['env_steps_per_launch'] != env_steps_per_launch:
            return None
        c['stale'] = c.get('source_hash') != kernel_source_hash()
        return c
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (measured)'
    except Exception:
        return HBM_FALLBACK_GBS, 'B200_PROFILING.md fallback'


def run_gpu_arm(a):
    cpu = None
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    if world == 1 and rank == 0 and not a.no_cpu_baseline:
        # before CUDA is initialised (fork-safe); bounded sample of the same workload
        v, cores, steps, wall = cpu_env_steps_per_sec(a.env_id, a.cpu_seconds)
        cpu = {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port',
               'sample': f'{steps} env-steps of {a.env_id} (defaults, U(-1,1) actions, auto-reset) in '
                         f'{wall:.1f} s wall: {cores} processes x one numpy oracle env each'}

    import torch
    from phoenix_drone_simulation_b200 import VecEnv
    ctx = DistCtx(a.gpus)
    assert ctx.world == a.gpus, f'--gpus {a.gpus} but WORLD_SIZE={ctx.world} (launch with torchrun for N>1)'
    dev = ctx.device
    n = a.num_envs
    env = VecEnv(a.env_id, n, device=dev, dtype=torch.float32, seed=a.seed, env_offset=ctx.rank * n)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(1234 + ctx.rank)
    seg_bytes = a.inner * n * (16 + env.obs_dim * 4)
    seg = Segment(env, a.inner, ring_slots(seg_bytes), gen, a.mode)

    sampler = ClockSampler(ctx.local_rank)
    ms, launches = time_device(env, seg, a.steps, a.warmup, ctx, sampler, per_step=a.launches)
    clocks = sampler.stop()
    if a.dump_outputs and ctx.rank == 0:
        # the ring still holds the last launch of the timed window: the final `inner` env.steps of the last step
        dump_outputs(seg, (a.warmup + a.steps) * a.launches - 1, a.dump_outputs)
    env_steps = a.steps * a.launches * a.inner * n * ctx.world
    value = env_steps / (ms * 1e-3)

    # roofline of the dominant kernel (the fused step).  The kernel is bound by ISSUE SLOTS, not by HBM:
    #   achieved = warp instructions per launch (ncu smsp__inst_executed.sum of this very launch shape, read
    #              from profiles/ together with the hash of the kernel sources it was captured from)
    #              / mean launch duration measured here with CUDA events
    #   peak     = SMs x 4 schedulers x SM clock under load (one warp instruction per scheduler and cycle)
    # The HBM view of the same launch (algorithmic bytes / duration against the measured copy bandwidth)
    # is reported next to it under `hbm`.
    peak, peak_src = measured_peak()
    steps_per_launch = a.steps * a.launches * a.inner // launches
    bytes_per_launch = env.rollout_bytes(steps_per_launch) * n
    us_per_launch = ms * 1e3 / launches
    achieved = bytes_per_launch / (us_per_launch * 1e-6) / 1e9
    counters = profile_counters(steps_per_launch * n)
    props = torch.cuda.get_device_properties(dev)
    sm_mhz = clocks['sm_mhz'] or 1965
    issue_peak = props.multi_processor_count * 4 * sm_mhz * 1e6
    hbm = {'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'peak_source': peak_src,
           'algorithmic_bytes_per_launch': bytes_per_launch,
           'bytes_per_env_step': bytes_per_launch / (steps_per_launch * n)}
    if counters:
        inst = counters['smsp__inst_executed.sum']
        ach_i = inst / (us_per_launch * 1e-6)
        roofline = {'bound': 'issue', 'achieved': ach_i / 1e9, 'peak': issue_peak / 1e9, 'unit': 'G warp-inst/s',
                    'frac': ach_i / issue_peak, 'traffic': counters['dram_bytes_read'] + counters['dram_bytes_write'],
                    'warp_inst_per_launch': inst, 'warp_inst_per_warp_step': inst / (steps_per_launch * n / 32),
                    'counters_source': counters['source'], 'counters_stale': counters['stale'],
                    'peak_source': f'{props.multi_processor_count} SMs x 4 schedulers x {sm_mhz} MHz (median SM clock under load)'}
    else:
        roofline = dict(hbm, bound='hbm', traffic=None)
    # SURVEY 8(d) sized the path as HBM-bound with the state read and written on EVERY env.step (542 B per env-step
    # for Hover-Simple H=2, ceiling = peak / 542 B): the fused launch keeps the state in registers across its steps,
    # which is why the line above is bounded by issue slots instead.  Reported for reference, not as the roofline.
    per_step_stream = {'bytes_per_env_step': 542, 'ceiling_env_steps_per_s': hbm['peak'] * 1e9 / 542,
                       'achieved_over_ceiling': (steps_per_launch * n / (us_per_launch * 1e-6)) / (hbm['peak'] * 1e9 / 542),
                       'what': 'SURVEY 8(d): state streamed through HBM on every env.step (a per-step kernel could not exceed this)'}
    roofline.update({'per_step_streaming': per_step_stream})
    roofline.update({'hbm': hbm, 'kernel': 'pdx::k_rollout<float, hover, simple, noise, philox>',
                     'env_steps_per_launch': steps_per_launch * n, 'us_per_launch': us_per_launch})

    # e2e: one bench step = the same a.launches x a.inner env.steps per environment, in 8-step chunks
    e2e_k = max(1, a.steps // a.e2e_div)
    e2e_ms, h2d, d2h = time_e2e(env, a.inner, e2e_k * a.launches, min(a.warmup, 3), ctx, 99 + ctx.rank)
    h2d, d2h = h2d * a.launches, d2h * a.launches
    e2e_steps = e2e_k * a.launches * a.inner * n * ctx.world
    link = link_ceiling(ctx.device, ctx)
    e2e_d2h_gbs = d2h * e2e_k / (e2e_ms * 1e-3) / 1e9            # per rank
    e2e = {'value': e2e_steps / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
           'numa_node_rank0': ctx.numa_node,
           'link': dict(link, achieved_d2h_gbs_per_rank=e2e_d2h_gbs, frac_of_d2h_ceiling=e2e_d2h_gbs / link['d2h_with_h2d_gbs'],
                        what='pinned-memory copy ceiling of this box with all ranks copying at once, per rank (measured here)'),
           'api': 'VecEnv.step_many_host: pinned host action/obs/reward/cost/flag buffers, H2D + launch + D2H per 8-step chunk on three streams, all inside the timed region'}

    extra = {}
    if ctx.world == 1:
        # the other action distribution SURVEY 8d asks for: a near-hover fixed policy (fewer resets)
        seg.actions = None
        segh = Segment(env, a.inner, ring_slots(seg_bytes), gen, a.mode, near_hover=True)
        kh = max(2, a.steps // 4)
        msh, _ = time_device(env, segh, kh, min(a.warmup, 2), ctx, per_step=a.launches)
        extra['fixed_policy'] = {'actions': 'HOVER_ACTION + N(0, 0.05)', 'value': kh * a.launches * a.inner * n / (msh * 1e-3),
                                 'unit': UNIT}
        del segh
    if a.large_envs and ctx.world == 1:
        # same kernel where the state cannot stay in L2: the honest HBM-bound measurement
        nl = a.large_envs
        big = VecEnv(a.env_id, nl, device=dev, dtype=torch.float32, seed=a.seed + 1)
        big.reset()
        inner_l = 8
        segl = Segment(big, inner_l, 2, gen, a.mode)
        kl = max(4, a.steps // 8)
        msl, ll = time_device(big, segl, kl, 3, ctx)
        usl = msl * 1e3 / ll
        spl = kl * inner_l // ll
        ach = big.rollout_bytes(spl) * nl / (usl * 1e-6) / 1e9
        extra['roofline_hbm_resident_off'] = {
            'envs': nl, 'state_bytes': int(big.state.numel() * 4), 'env_steps_per_launch': spl * nl,
            'us_per_launch': usl, 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
            'env_steps_per_s': kl * inner_l * nl / (msl * 1e-3)}
        del big, segl
    if ctx.world == 1 and not a.no_ppo_rollout:
        try:
            extra['ppo_rollout'] = ppo_rollout_leg(dev)
        except Exception as e:                       # never lose the headline line to the companion leg
            extra['ppo_rollout'] = {'error': repr(e)[:200]}

    episodes = int(ctx.episodes.item()) if ctx.dist else int(env.episode_stats()[0].item())
    ctx.close()
    if ctx.rank != 0:
        return
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup,
        'ms_per_step': ms / a.steps, 'timed_region_ms': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(a, n),
        'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline,
        'episodes_finished': episodes,
    }
    if cpu:
        line['cpu_baseline'] = cpu
    line.update(extra)
    print(json.dumps(line), flush=True)


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=20)
    p.add_argument('--launches', type=int, default=16, help='fused launches (rollout segments) per bench step')
    p.add_argument('--warmup', type=int, default=5)
    p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    p.add_argument('--env-id', default=ENV_ID)
    p.add_argument('--num-envs', type=int, default=65536, help='environments per GPU')
    p.add_argument('--inner', type=int, default=64, help='env.steps per bench step (rollout segment)')
    p.add_argument('--mode', default='fused', choices=['fused', 'per-step'])
    p.add_argument('--seed', type=int, default=0)
    p.add_argument('--cpu-seconds', type=float, default=10.0)
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--e2e-div', type=int, default=4, help='e2e leg times steps/e2e_div segments')
    p.add_argument('--large-envs', type=int, default=4 * 1024 * 1024)
    p.add_argument('--no-ppo-rollout', action='store_true', help='skip the configs[4] companion leg')
    p.add_argument('--dump-outputs', metavar='DIR',
                   help='after the timed steps, write what the last launch of the last step returned (obs, reward, cost, '
                        'terminated, truncated of a fixed, seeded sample of environments) as DIR/<name>.npy, float32')
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and a.impl == 'reference':
        p.error('--dump-outputs writes the outputs of the CUDA engine (--impl b200)')
    if a.impl == 'reference':
        run_reference_arm(a)
    else:
        run_gpu_arm(a)


if __name__ == '__main__':
    main()
