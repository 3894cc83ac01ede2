#!/usr/bin/env python
"""NPG and TRPO epoch phases with update_kernel='torch' vs 'cuda' on the recorded training shape of
tools/bench_ppo_update.py (DroneCircleBulletEnv-v0, 16,384 envs x 64 steps, cg_iters 10, target_kl 0.01).

    python tools/bench_npg_update.py [--env DroneCircleBulletEnv-v0 --envs 16384 --steps 64 --reps 3]

One object per (algorithm, update kernel), epochs alternated after one warm-up epoch each.  CUDA events time the
rollout, the value phase and the policy phase, the latter split into the surrogate gradient, the conjugate-gradient
solve (CG, x^T F x and the step) and the step-size search (NPG: none; TRPO: the line search).  Then pdx_ppo_pi_fvp alone
on every 4th row of one batch against the FP32 floor of its arithmetic, 3 D h1 + 5 h1 h2 + 21 h2 FMAs per sample at
SMs x 128 lanes x 2 FLOP x the maximum SM clock.  Prints JSON lines, the card's name, power limit and clock first.
"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from bench_ppo_update import gpu_info  # noqa: E402


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--env', default='DroneCircleBulletEnv-v0')
    p.add_argument('--envs', type=int, default=16384)
    p.add_argument('--steps', type=int, default=64)
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--kernel-reps', type=int, default=50)
    a = p.parse_args()
    from phoenix_drone_simulation_b200.npg import KL_SCALE, NPG
    from phoenix_drone_simulation_b200.ppo import pi_flat_params, pi_fvp
    from phoenix_drone_simulation_b200.trpo import TRPO
    info = gpu_info()
    print(json.dumps(info), flush=True)
    algs = {(n, k): c(a.env, num_envs=a.envs, steps=a.steps, epochs=1000, seed=0, update_kernel=k)
            for n, c in (('npg', NPG), ('trpo', TRPO)) for k in ('torch', 'cuda')}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def epoch(alg):
        marks = {}
        for name in ('update_v', 'update_pi', '_surrogate_grad', 'search_step_size'):
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
        e3.record()
        torch.cuda.synchronize()
        alg.epoch += 1
        t = lambda m: marks[m][0].elapsed_time(marks[m][1])
        ms = {'rollout': e0.elapsed_time(e1), 'value_phase': t('update_v'), 'policy_phase': t('update_pi'),
              'gradient': t('_surrogate_grad'), 'cg': marks['_surrogate_grad'][1].elapsed_time(marks['search_step_size'][0]),
              'step_size_search': t('search_step_size'), 'update': e1.elapsed_time(e2), 'epoch': e0.elapsed_time(e3)}
        return ms, upd, data

    for alg in algs.values():                                # warm-up: module loads, allocator, cuBLAS heuristics
        epoch(alg)
    rows = {k: [] for k in algs}
    for _ in range(a.reps):
        for k, alg in algs.items():
            ms, upd, data = epoch(alg)
            rows[k].append((ms, upd))
    T, N = a.steps, a.envs
    for (n, k), rs in rows.items():
        med = {f: statistics.median(r[0][f] for r in rs) for f in rs[0][0]}
        print(json.dumps({'alg': n, 'update_kernel': k, 'reps': a.reps, **{f'{f}_ms': round(v, 3) for f, v in med.items()},
                          'epoch_fps': round(T * N / (med['epoch'] / 1e3)),
                          'accept_step': [r[1]['accept_step'] for r in rs]}), flush=True)

    # ---- the Fisher-vector product alone on every 4th row of one batch
    alg = algs[('npg', 'cuda')]
    obs = alg.ac.obs_oms(data['obs'].reshape(T * N, -1).float()).contiguous()
    idx = torch.arange(0, obs.shape[0], 4, device=obs.device)
    v = torch.randn_like(pi_flat_params(alg.ac))
    out = torch.empty_like(v)
    for _ in range(3):
        pi_fvp(alg.ac, obs, v, 0.1, KL_SCALE, index=idx, out=out)
    s, e = ev(), ev()
    s.record()
    for _ in range(a.kernel_reps):
        pi_fvp(alg.ac, obs, v, 0.1, KL_SCALE, index=idx, out=out)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / a.kernel_reps
    lins = [m for m in alg.ac.pi if isinstance(m, torch.nn.Linear)]
    D, h1, h2 = lins[0].in_features, lins[0].out_features, lins[1].out_features
    fma = 3 * D * h1 + 5 * h1 * h2 + 21 * h2
    flop = 2.0 * fma * idx.numel()
    res = {'fvp_kernel_ms': round(ms, 4), 'samples': idx.numel(), 'fma_per_sample': fma,
           'gflop_per_call': round(flop / 1e9, 3), 'achieved_tflops': round(flop / (ms / 1e3) / 1e12, 2)}
    if info.get('max_sm_clock_mhz'):
        peak = info['sms'] * 128 * 2 * info['max_sm_clock_mhz'] * 1e6
        res.update({'fp32_peak_tflops': round(peak / 1e12, 1), 'floor_ms': round(flop / peak * 1e3, 4),
                    'fraction_of_fp32_floor': round(flop / peak * 1e3 / ms, 3)})
    print(json.dumps(res), flush=True)


if __name__ == '__main__':
    main()
