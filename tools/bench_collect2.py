import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from phoenix_drone_simulation_b200 import VecEnv
from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
env_id, kernel = sys.argv[1], sys.argv[2]
for n in [int(x) for x in sys.argv[3].split(',')]:
    for T in (16, 64):
        torch.manual_seed(0)
        env = VecEnv(env_id, n, seed=2, keep_final_obs=True)
        ac = ActorCritic(env.obs_dim, policy_kernel=kernel)
        col = RolloutCollector(env, ac, T)
        for _ in range(2):
            col.collect()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            col.collect()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        print(json.dumps({'env': env_id, 'k': kernel, 'fused': col.fused_used, 'n': n, 'T': T, 'ms': round(ms, 3), 'Gsteps': round(T * n / ms / 1e6, 3)}), flush=True)
        del env, ac, col
