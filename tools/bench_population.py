"""One PopulationPPO(update_kernel='cuda') epoch of P members against P sequential PPO(update_kernel='cuda') epochs of
the same per-member shape -- what a seed sweep does today.

    python tools/bench_population.py [--members 1 8 64] [--envs 512] [--steps 64] [--repeats 5] [--json out.json]

DroneHoverBulletEnv-v0 with iwpg.py's defaults (32 k samples per member and epoch at 512 x 64).  Reports the rollout,
value-phase, policy-phase and whole-epoch times (ms; medians over repeats that alternate the two forms after one warm-up
epoch each) and member-epochs per second.  Device events, synchronised per phase.  Prints the card name and power
limit with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from phoenix_drone_simulation_b200.population import PopulationPPO  # noqa: E402
from phoenix_drone_simulation_b200.ppo import PPO  # noqa: E402

ENV = 'DroneHoverBulletEnv-v0'


def _phases(collect, update_v, update_pi, finish):
    """(rollout, value, policy, epoch) ms of one epoch."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev[0].record()
    data = collect()
    ev[1].record()
    update_v(data)
    ev[2].record()
    update_pi(data)
    ev[3].record()
    finish(data)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    return [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), wall]


def population_epoch(pop):
    state = {}

    def update_v(data):
        obs = pop._member_major(data['obs'].float())
        state['obs'] = (obs - pop.obs_mean.unsqueeze(1)) / (pop.obs_std.unsqueeze(1) + pop.obs_eps)
        pop.update_v(state['obs'], pop._member_major(data['target_v']))

    def update_pi(data):
        pop.update_pi(state['obs'], pop._member_major(data['act']), pop._member_major(data['adv']),
                      pop._member_major(data['log_p']))

    def finish(data):
        pop.update_running_statistics(data)
        pop.epoch += 1
    pop.log_std.fill_(-0.7)
    return _phases(pop.collect, update_v, update_pi, finish)


def sequential_epochs(algs):
    """The P single-agent epochs back to back, phases summed over the agents."""
    tot = [0.0] * 4
    for alg in algs:
        state = {}

        def update_v(data, alg=alg):
            T, N = data['rew'].shape
            state['obs'] = alg.ac.obs_oms(data['obs'].reshape(T * N, -1).float())
            alg.update_v(state['obs'], data['target_v'].reshape(-1))

        def update_pi(data, alg=alg):
            T, N = data['rew'].shape
            alg.update_pi(state['obs'], data['act'].reshape(T * N, -1), data['adv'].reshape(-1),
                          data['log_p'].reshape(-1))

        def finish(data, alg=alg):
            alg.collector.update_running_statistics(data)
            alg.sched.step()
            alg.epoch += 1
        for k, v in enumerate(_phases(alg.collector.collect, update_v, update_pi, finish)):
            tot[k] += v
    return tot


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        q = torch.cuda.get_device_name()
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, nargs='+', default=[1, 8, 64])
    ap.add_argument('--envs', type=int, default=512)
    ap.add_argument('--steps', type=int, default=64)
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_population needs a CUDA device')
    results = {'card': card(), 'env': ENV, 'envs_per_member': a.envs, 'steps': a.steps, 'rows': []}
    print(results['card'], flush=True)
    kw = dict(steps=a.steps, epochs=1000, update_kernel='cuda')
    for P in a.members:
        pop = PopulationPPO(ENV, members=P, num_envs_per_member=a.envs, seed=0, **kw)
        algs = [PPO(ENV, num_envs=a.envs, seed=m, **kw) for m in range(P)]
        for alg in algs:
            alg.ac.set_log_std(0.5)
        population_epoch(pop)                            # warm-up: module loads, allocations, scratch
        sequential_epochs(algs)
        pops, seqs = [], []
        for _ in range(a.repeats):
            pops.append(population_epoch(pop))
            seqs.append(sequential_epochs(algs))
        med = lambda rows: [statistics.median(r[k] for r in rows) for k in range(4)]
        mp, ms = med(pops), med(seqs)
        row = {'members': P,
               'population_ms': dict(zip(('rollout', 'value', 'policy', 'epoch'), [round(x, 2) for x in mp])),
               'sequential_ms': dict(zip(('rollout', 'value', 'policy', 'epoch'), [round(x, 2) for x in ms])),
               'population_member_epochs_per_s': round(P / mp[3] * 1e3, 2),
               'sequential_member_epochs_per_s': round(P / ms[3] * 1e3, 2),
               'speedup': round(ms[3] / mp[3], 2)}
        results['rows'].append(row)
        print(json.dumps(row), flush=True)
        del pop, algs
        torch.cuda.empty_cache()
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, 'w') as f:
            json.dump(results, f, indent=1)


if __name__ == '__main__':
    main()
