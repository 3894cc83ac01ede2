#!/usr/bin/env python
"""PPO epoch phases with update_kernel='torch' vs 'cuda' on the recorded training shape (BASELINE.md "PPO training
FPS": DroneCircleBulletEnv-v0, 16,384 envs x 64 steps, the iwpg.py defaults: 80 full-batch policy steps, 5 x 16
value mini-batch steps).

    python tools/bench_ppo_update.py [--env DroneCircleBulletEnv-v0 --envs 16384 --steps 64 --reps 3]

One PPO object per update kernel, epochs alternated A/B after one warm-up epoch each.  CUDA events time the rollout,
the value phase, the policy phase, the whole update() and the whole epoch (rollout + update + running statistics).
Then pdx_ppo_pi_grad alone on one full batch, against the FP32 floor of its arithmetic: per sample
D h1 + h1 h2 + 4 h2 FMAs forward, 4 h2 + h1 h2 backward, D h1 + h1 h2 + 4 h2 weight gradients, at
SMs x 128 lanes x 2 FLOP x the maximum SM clock.  Prints JSON lines.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402


def gpu_info():
    info = {'gpu': torch.cuda.get_device_name(0), 'sms': torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits',
                            '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        info['power_limit_w'], info['max_sm_clock_mhz'] = float(q[0]), float(q[1])
    except Exception as e:                                   # the numbers are then reported without it
        info['power_limit_w'] = info['max_sm_clock_mhz'] = None
        info['nvidia_smi'] = repr(e)
    return info


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--env', default='DroneCircleBulletEnv-v0')
    p.add_argument('--envs', type=int, default=16384)
    p.add_argument('--steps', type=int, default=64)
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--kernel-reps', type=int, default=20)
    a = p.parse_args()
    from phoenix_drone_simulation_b200.ppo import PPO, pi_loss_and_grad
    info = gpu_info()
    print(json.dumps(info), flush=True)
    algs = {k: PPO(a.env, num_envs=a.envs, steps=a.steps, epochs=1000, seed=0, update_kernel=k) for k in ('torch', 'cuda')}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def epoch(alg):
        marks = {}
        for name in ('update_v', 'update_pi'):
            f = getattr(type(alg), name)

            def wrapped(*args, _f=f, _n=name):
                s, e = ev(), ev()
                s.record()
                r = _f(alg, *args)
                e.record()
                marks[_n] = (s, e)
                return r
            setattr(alg, name, wrapped)
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        if alg.use_exploration_noise_anneal:
            alg.ac.set_log_std(1 - alg.epoch / max(1, alg.epochs))
        e0.record()
        data = alg.collector.collect()
        e1.record()
        upd = alg.update(data)
        e2.record()
        alg.collector.update_running_statistics(data)
        if alg.sched is not None:
            alg.sched.step()
        e3.record()
        torch.cuda.synchronize()
        alg.epoch += 1
        ms = {'rollout': e0.elapsed_time(e1), 'value_phase': marks['update_v'][0].elapsed_time(marks['update_v'][1]),
              'policy_phase': marks['update_pi'][0].elapsed_time(marks['update_pi'][1]), 'update': e1.elapsed_time(e2),
              'epoch': e0.elapsed_time(e3)}
        return ms, upd, data

    for k in algs:                                           # warm-up: module loads, allocator, cuBLAS heuristics
        epoch(algs[k])
    rows = {k: [] for k in algs}
    for _ in range(a.reps):
        for k in algs:
            ms, upd, data = epoch(algs[k])
            rows[k].append(ms)
    T, N = a.steps, a.envs
    summary = {}
    for k, rs in rows.items():
        med = {f: statistics.median(r[f] for r in rs) for f in rs[0]}
        summary[k] = med
        print(json.dumps({'update_kernel': k, 'reps': a.reps, **{f'{f}_ms': round(v, 3) for f, v in med.items()},
                          'epoch_fps': round(T * N / (med['epoch'] / 1e3)), 'pi_iters': upd['pi_iters']}), flush=True)
    print(json.dumps({'speedup_update': round(summary['torch']['update'] / summary['cuda']['update'], 2),
                      'speedup_policy_phase': round(summary['torch']['policy_phase'] / summary['cuda']['policy_phase'], 2),
                      'speedup_value_phase': round(summary['torch']['value_phase'] / summary['cuda']['value_phase'], 2),
                      'speedup_epoch': round(summary['torch']['epoch'] / summary['cuda']['epoch'], 2)}), flush=True)

    # ---- the policy kernel alone on one full batch
    alg = algs['cuda']
    obs = alg.ac.obs_oms(data['obs'].reshape(T * N, -1).float()).contiguous()
    act, adv = data['act'].reshape(T * N, -1).contiguous(), data['adv'].reshape(-1).contiguous()
    logp_old = data['log_p'].reshape(-1).contiguous()
    for _ in range(3):
        pi_loss_and_grad(alg.ac, obs, act, adv, logp_old, alg.clip_ratio)
    s, e = ev(), ev()
    s.record()
    for _ in range(a.kernel_reps):
        pi_loss_and_grad(alg.ac, obs, act, adv, logp_old, alg.clip_ratio)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / a.kernel_reps
    lins = [m for m in alg.ac.pi if isinstance(m, torch.nn.Linear)]
    D, h1, h2 = lins[0].in_features, lins[0].out_features, lins[1].out_features
    fma = 2 * (D * h1 + h1 * h2 + 4 * h2) + (4 * h2 + h1 * h2)
    flop = 2.0 * fma * T * N
    out = {'policy_kernel_ms': round(ms, 4), 'samples': T * N, 'fma_per_sample': fma, 'gflop_per_step': round(flop / 1e9, 2),
           'achieved_tflops': round(flop / (ms / 1e3) / 1e12, 2)}
    if info.get('max_sm_clock_mhz'):
        peak = info['sms'] * 128 * 2 * info['max_sm_clock_mhz'] * 1e6
        out.update({'fp32_peak_tflops': round(peak / 1e12, 1), 'floor_ms': round(flop / peak * 1e3, 4),
                    'fraction_of_fp32_floor': round(flop / peak * 1e3 / ms, 3)})
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
