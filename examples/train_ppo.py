#!/usr/bin/env python
"""On-policy training (PPO, IWPG, NPG or TRPO) on the batched engine, one process per GPU.

    python examples/train_ppo.py --env DroneHoverSimpleEnv-v0 --epochs 30
    python examples/train_ppo.py --alg trpo --update-kernel cuda
    python examples/train_ppo.py --population 8 --num-envs 512 --update-kernel cuda    # seeds 0..7 in one process
    python examples/train_ppo.py --population 4 --alg trpo --update-kernel cuda
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 examples/train_ppo.py --epochs 30

Counterpart of `python -m phoenix_drone_simulation.train --alg {ppo,iwpg,npg,trpo} --env <id> --cores N`
(train.py:97-149 of the reference): environments shard over the GPUs by global index, gradients,
the observation normaliser and the episode statistics are all-reduced over NCCL, and -- like the
reference's check_distributed_parameters (algs/iwpg/iwpg.py:228-237) -- the ranks verify at the end
that their parameters are identical.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--alg', default='ppo', choices=['ppo', 'iwpg', 'npg', 'trpo'],
                   help="iwpg: PPO's loop with the unclipped surrogate; npg / trpo: conjugate-gradient policy steps")
    p.add_argument('--env', default='DroneHoverSimpleEnv-v0')
    p.add_argument('--epochs', type=int, default=30)
    p.add_argument('--num-envs', type=int, default=4096, help='per GPU')
    p.add_argument('--steps', type=int, default=64)
    p.add_argument('--seed', type=int, default=0)
    p.add_argument('--update-kernel', default='torch', choices=['torch', 'cuda'],
                   help="'cuda': losses, gradients (and NPG / TRPO's Fisher-vector products) of the update in the fused "
                        "kernels pdx_ppo_pi_grad / pdx_ppo_v_grad / pdx_ppo_pi_fvp")
    p.add_argument('--population', type=int, default=0,
                   help='train this many agents of --alg (seeds seed .. seed + P - 1, --num-envs environments each) in one '
                        'process on one GPU (population.PopulationPPO / PopulationNPG / PopulationTRPO); prints one row '
                        'per member and epoch')
    a = p.parse_args()
    if a.population:
        if int(os.environ.get('WORLD_SIZE', '1')) > 1:
            p.error('--population trains on one GPU: start it once per GPU, not under torch.distributed.run')
        from phoenix_drone_simulation_b200.population import PopulationNPG, PopulationPPO, PopulationTRPO
        cls, kw = {'ppo': (PopulationPPO, {}), 'iwpg': (PopulationPPO, {'clip_ratio': None}), 'npg': (PopulationNPG, {}),
                   'trpo': (PopulationTRPO, {})}[a.alg]
        pop = cls(a.env, members=a.population, num_envs_per_member=a.num_envs, steps=a.steps, epochs=a.epochs,
                  seed=a.seed, update_kernel=a.update_kernel, **kw)
        keys = ('EpRet', 'EpLen', 'episodes', 'loss_pi', 'loss_v', 'kl')
        keys += ('accept_step', 'xHx') if a.alg in ('npg', 'trpo') else ('pi_iters',)
        for _ in range(a.epochs):
            row = pop.learn_one_epoch()
            for m in range(pop.P):
                print(json.dumps({'epoch': row['epoch'], 'member': m, 'seed': a.seed + m, 'FPS': round(row['FPS'], 1),
                                  **{k: (round(row[k][m], 4) if isinstance(row[k][m], float) else row[k][m])
                                     for k in keys}}),
                      flush=True)
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get('NCCL_DEBUG') and not os.environ.get('NCCL_DEBUG_FILE'):
            os.environ['NCCL_DEBUG_FILE'] = '/dev/stderr'     # stdout carries the JSON lines
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from phoenix_drone_simulation_b200.npg import NPG
    from phoenix_drone_simulation_b200.ppo import PPO
    from phoenix_drone_simulation_b200.trpo import TRPO
    cls, kw = {'ppo': (PPO, {}), 'iwpg': (PPO, {'clip_ratio': None}), 'npg': (NPG, {}), 'trpo': (TRPO, {})}[a.alg]
    alg = cls(a.env, num_envs=a.num_envs, steps=a.steps, epochs=a.epochs, device=f'cuda:{local}', seed=a.seed, dist=dist,
              update_kernel=a.update_kernel, **kw)
    for _ in range(a.epochs):
        row = alg.learn_one_epoch()
        if rank == 0:
            print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in row.items()}), flush=True)
    # all ranks must hold the same networks (sync by construction: same init, averaged gradients)
    chk = torch.stack([sum(p_.double().sum() for p_ in alg.ac.pi.parameters()),
                       sum(p_.double().sum() for p_ in alg.ac.v.parameters()),
                       alg.ac.obs_oms.mean.double().sum(), alg.ac.obs_oms.std.double().sum()])
    if world > 1:
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), f'ranks diverged: {lo.tolist()} vs {hi.tolist()}'
        if rank == 0:
            print(json.dumps({'ranks': world, 'parameters_identical_across_ranks': True}), flush=True)
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
