"""Fixed-policy evaluation at the scale of the reference's experiment 07 (3 control modes x 162 runs, SURVEY §6):
per control mode, 162 policies x 128 episodes on DroneCircleBulletEnv-v0 (PWM agg 2, AttitudeRate agg 4, Attitude
agg 8), the policies built from the two KAT models of that mode (tests/golden_collector/kat_models) with perturbed
weights.  One JSON line per mode:
  * evaluate_many (one pdx_evaluate launch): synchronised wall time of the call, kernel time (torch.profiler, a
    pass of its own), executed env-steps (sum of the episode lengths) and env-steps/s;
  * the host loop of policy_io.evaluate on the first 8 policies, and that time scaled by 162 / 8 (a scaling, not a
    measurement of 162 policies);
  * diagnostic against evaluate(policy_kernel='cuda') on those 8 policies at full length: the fraction of episodes
    with equal length and the largest |return difference| (the two step instantiations differ in the last bits,
    which a 500-step chaotic rollout may amplify).
    python tools/bench_evaluate.py [--env DroneHoverBulletEnv-v0] [--policies 162] [--episodes 128] [--repeats 3]"""
import argparse
import glob
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from phoenix_drone_simulation_b200 import VecEnv
from phoenix_drone_simulation_b200.policy_io import evaluate, evaluate_many, load_policy_json
from phoenix_drone_simulation_b200.rollout import ActorCritic

MODES = {'DroneCircleBulletEnv-v0': [('PWM', 2), ('AttitudeRate', 4), ('Attitude', 8)],
         'DroneHoverBulletEnv-v0': [('PWM', None)]}
KAT = os.path.join(ROOT, 'tests', 'golden_collector', 'kat_models')


def policies_for(env_id, mode, n, kernel='cuda'):
    """The KAT models of `mode` and perturbed copies of them; for ids whose observation width differs from the
    KAT models' (Hover: 34), randomly initialised policies."""
    files = sorted(glob.glob(os.path.join(KAT, f'{mode}_seed_*_model.json')))
    obs_dim = VecEnv(env_id, 1, control_mode=mode).obs_dim
    if load_policy_json(files[0], device='cpu').pi.net[0].in_features != obs_dim:
        out = []
        for k in range(n):
            torch.manual_seed(k)
            out.append(ActorCritic(obs_dim, policy_kernel=kernel))
        return out
    out = []
    for k in range(n):
        ac = load_policy_json(files[k % len(files)], policy_kernel=kernel)
        if k >= len(files):                           # the KAT models themselves, then perturbed copies
            g = torch.Generator(device='cuda').manual_seed(k)
            with torch.no_grad():
                for m in ac.pi:
                    if isinstance(m, torch.nn.Linear):
                        m.weight.add_(0.05 * m.weight.std() * torch.randn(m.weight.shape, device='cuda', generator=g))
        out.append(ac)
    return out


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return {'gpu': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip().splitlines()[torch.cuda.current_device()]
            if q.returncode == 0 else 'unavailable'}


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if 'k_evaluate' in e.key) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--env', default='DroneCircleBulletEnv-v0', choices=sorted(MODES))
    ap.add_argument('--policies', type=int, default=162)
    ap.add_argument('--episodes', type=int, default=128)
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--loop-policies', type=int, default=8)
    a = ap.parse_args()
    info = gpu_info()
    for mode, agg in MODES[a.env]:
        kw = dict(control_mode=mode) if agg is None else dict(control_mode=mode, aggregate_phy_steps=agg)
        pols = policies_for(a.env, mode, a.policies)
        run = lambda: evaluate_many(a.env, pols, a.episodes, seed=0, **kw)
        run()                                                   # warm-up: module load, shared-memory opt-in
        walls = []
        for _ in range(a.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ret, length, cost = run()                           # returns host arrays: ends in a synchronise
            walls.append(time.perf_counter() - t0)
        k_ms = kernel_ms(run)
        steps = int(length.sum())
        # the host loop of evaluate on a subset
        sub = pols[:a.loop_policies]
        evaluate(a.env, sub[0], a.episodes, seed=0, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop = [evaluate(a.env, ac, a.episodes, seed=0, **kw) for ac in sub]
        loop_s = time.perf_counter() - t0
        eq_len = float(np.mean([np.mean(l[1] == length[k]) for k, l in enumerate(loop)]))
        d_ret = float(max(np.abs(l[0] - ret[k]).max() for k, l in enumerate(loop)))
        wall = float(np.median(walls))
        print(json.dumps({
            'env_id': a.env, 'control_mode': mode, 'agg': agg, 'policies': a.policies, 'episodes': a.episodes,
            'evaluate_many_wall_s': wall, 'evaluate_many_wall_s_all': walls, 'kernel_ms': k_ms,
            'env_steps': steps, 'env_steps_per_s_wall': steps / wall, 'env_steps_per_s_kernel': steps / (k_ms * 1e-3),
            'mean_length': float(length.mean()), 'mean_return': float(ret.mean()),
            'evaluate_loop_policies': len(sub), 'evaluate_loop_wall_s': loop_s,
            'evaluate_loop_wall_s_scaled_to_all_policies': loop_s * a.policies / len(sub),
            'diag_equal_length_fraction': eq_len, 'diag_max_abs_return_diff': d_ret, **info}), flush=True)


if __name__ == '__main__':
    main()
