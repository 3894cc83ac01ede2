"""One PopulationPPO(update_kernel='cuda') epoch of P members against P sequential PPO(update_kernel='cuda') epochs of
the same per-member shape -- what a seed sweep does today.  --alg npg / trpo: PopulationNPG / PopulationTRPO against
P sequential NPG / TRPO agents, the policy phase also split into the surrogate gradient, the conjugate-gradient solve
(CG, x^T F x and the step) and the step-size search (NPG: none; TRPO: the line search), as tools/bench_npg_update.py.

    python tools/bench_population.py [--alg ppo] [--members 1 8 64] [--envs 512] [--steps 64] [--repeats 5] [--json out.json]

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

from phoenix_drone_simulation_b200.npg import NPG  # noqa: E402
from phoenix_drone_simulation_b200.population import PopulationNPG, PopulationPPO, PopulationTRPO  # noqa: E402
from phoenix_drone_simulation_b200.ppo import PPO  # noqa: E402
from phoenix_drone_simulation_b200.trpo import TRPO  # noqa: E402

ENV = 'DroneHoverBulletEnv-v0'
ALGS = {'ppo': (PopulationPPO, PPO), 'npg': (PopulationNPG, NPG), 'trpo': (PopulationTRPO, TRPO)}
SPLIT = ('gradient', 'cg', 'search')


def _instrument(obj):
    """Wraps obj's _surrogate_grad and search_step_size (NPG / TRPO) in CUDA events; returns the dict they fill."""
    marks = {}
    for name in ('_surrogate_grad', 'search_step_size'):
        f = getattr(type(obj), name)

        def wrapped(*args, _f=f, _n=name):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = _f(obj, *args)
            e.record()
            marks[_n] = (s, e)
            return r
        setattr(obj, name, wrapped)
    return marks


def _split(marks):
    """(gradient, cg, search) ms of the policy phase just timed."""
    g, s = marks['_surrogate_grad'], marks['search_step_size']
    return [g[0].elapsed_time(g[1]), g[1].elapsed_time(s[0]), s[0].elapsed_time(s[1])]


def _phases(collect, update_v, update_pi, finish, marks=None):
    """(rollout, value, policy, epoch) ms of one epoch, then the policy phase's split when `marks` is given."""
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
    out = [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), wall]
    return out + _split(marks) if marks is not None else out


def population_epoch(pop, marks=None):
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
    return _phases(pop.collect, update_v, update_pi, finish, marks)


def sequential_epochs(algs, marks=None):
    """The P single-agent epochs back to back, phases summed over the agents."""
    tot = [0.0] * (4 if marks is None else 7)
    for i, alg in enumerate(algs):
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
            if alg.sched is not None:                    # NPG / TRPO: no actor optimiser, no schedule
                alg.sched.step()
            alg.epoch += 1
        for k, v in enumerate(_phases(alg.collector.collect, update_v, update_pi, finish,
                                      None if marks is None else marks[i])):
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
    ap.add_argument('--alg', default='ppo', choices=sorted(ALGS))
    ap.add_argument('--members', type=int, nargs='+', default=[1, 8, 64])
    ap.add_argument('--envs', type=int, default=512)
    ap.add_argument('--steps', type=int, default=64)
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_population needs a CUDA device')
    results = {'card': card(), 'alg': a.alg, 'env': ENV, 'envs_per_member': a.envs, 'steps': a.steps, 'rows': []}
    print(results['card'], flush=True)
    kw = dict(steps=a.steps, epochs=1000, update_kernel='cuda')
    pop_cls, alg_cls = ALGS[a.alg]
    for P in a.members:
        pop = pop_cls(ENV, members=P, num_envs_per_member=a.envs, seed=0, **kw)
        algs = [alg_cls(ENV, num_envs=a.envs, seed=m, **kw) for m in range(P)]
        for alg in algs:
            alg.ac.set_log_std(0.5)
        pop_marks = seq_marks = None
        if a.alg != 'ppo':
            pop_marks, seq_marks = _instrument(pop), [_instrument(alg) for alg in algs]
        population_epoch(pop, pop_marks)                 # warm-up: module loads, allocations, scratch
        sequential_epochs(algs, seq_marks)
        pops, seqs = [], []
        for _ in range(a.repeats):
            pops.append(population_epoch(pop, pop_marks))
            seqs.append(sequential_epochs(algs, seq_marks))
        med = lambda rows: [statistics.median(r[k] for r in rows) for k in range(len(rows[0]))]
        mp, ms = med(pops), med(seqs)
        row = {'members': P,
               'population_ms': dict(zip(('rollout', 'value', 'policy', 'epoch'), [round(x, 2) for x in mp])),
               'sequential_ms': dict(zip(('rollout', 'value', 'policy', 'epoch'), [round(x, 2) for x in ms])),
               'population_member_epochs_per_s': round(P / mp[3] * 1e3, 2),
               'sequential_member_epochs_per_s': round(P / ms[3] * 1e3, 2),
               'speedup': round(ms[3] / mp[3], 2)}
        if a.alg != 'ppo':
            row['population_policy_split_ms'] = dict(zip(SPLIT, [round(x, 2) for x in mp[4:]]))
            row['sequential_policy_split_ms'] = dict(zip(SPLIT, [round(x, 2) for x in ms[4:]]))
            row['accept_step'] = pop.step_info['accept_step']
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
