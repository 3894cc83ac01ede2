"""k_rollout's launch shape depends on the shard size (pick_shape, csrc/pdx_dispatch.cuh): a shard that fits in one
wave is spread with the fewest warps on the busiest SM, so a VecEnv of n environments and the shards that split it
launch with different block sizes (from 16,384 environments up) and vote on reset-package regeneration in different
thread groups.  The results of
an environment depend on (seed, global env index, step counter) only; the vote group decides WHEN a package is
regenerated, never its contents.  So everything the kernel returns must be bit-identical, and so must every state
word except the pending-package bits of ep_index and the contents of package slots that are still pending.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

T_LAUNCH, LAUNCHES = 64, 2            # 128 env.steps: auto-resets and package regeneration both happen

CONFIGS = {
    'hover_simple': ('DroneHoverSimpleEnv-v0', {}),
    'circle_h8': ('DroneCircleSimpleEnv-v0', dict(observation_history_size=8)),    # row mode 2
    'takeoff_simple': ('DroneTakeOffSimpleEnv-v0', {}),
    'hover_bullet': ('DroneHoverBulletEnv-v0', {}),
}
SIZES = [1, 31, 447, 449, 16384, 65536, 65537, 75776]


def _vec(env_id, n, offset, kw):
    from phoenix_drone_simulation_b200 import VecEnv
    return VecEnv(env_id, n, seed=11, env_offset=offset, **kw)


def _shards(n):
    """(offset, size) of the launches that stand in for one launch of n environments, together covering
    [0, n).  A single environment has nothing to split: it is the first environment of a larger shard."""
    if n == 1:
        return [(0, 449)]
    k = n // 3
    return [(0, k), (k, n - k)]


def _run(env, actions):
    T, n = actions.shape[:2]
    dev, dt, D = env.device, env.dtype, env.obs_dim
    outs = []
    for _ in range(LAUNCHES):
        out = {'obs': torch.empty((T, n, D), dtype=dt, device=dev),
               'reward': torch.empty((T, n), dtype=dt, device=dev), 'cost': torch.empty((T, n), dtype=dt, device=dev),
               'terminated': torch.empty((T, n), dtype=torch.uint8, device=dev),
               'truncated': torch.empty((T, n), dtype=torch.uint8, device=dev),
               'final_obs': torch.zeros((T, n, D), dtype=dt, device=dev),
               'episode_return': torch.empty((T, n), dtype=dt, device=dev),
               'episode_length': torch.empty((T, n), dtype=torch.int32, device=dev)}
        outs.append(env.step_many(actions.contiguous(), out))
        actions = actions.flip(0)
    return outs


def _words(env):
    """Bit patterns of the state: per-environment planes [P, n, 4] (ep_index without its pending bits), the package
    pool [slots, n, words] and the pending mask [n]."""
    assert env.dtype == torch.float32                        # ep_index holds its bit pattern (csrc/pdx_layout.h)
    bits = env.state.view(torch.int32)
    fw, _ = env._field('ep_index')
    pool_w, pool_n = env._field('pool')
    planes = bits[:pool_w // 4].clone()
    _, pending = env.episode_counters()
    planes[fw // 4, :, fw % 4] &= ~15
    pool = bits[pool_w // 4:].reshape(-1).view(4, env.num_envs, -1)        # slot s of env j: ((s n + j) pack) quads
    assert pool.shape[2] * 4 == pool_n
    return planes, pool, pending


@pytest.mark.parametrize('n', SIZES)
@pytest.mark.parametrize('cfg', list(CONFIGS))
def test_shard_shapes_give_identical_results(cfg, n):
    env_id, kw = CONFIGS[cfg]
    full = _vec(env_id, n, 0, kw)
    parts = [_vec(env_id, m, off, kw) for off, m in _shards(n)]
    full.reset()
    for p in parts:
        p.reset()
    g = torch.Generator(device='cuda').manual_seed(5)
    n_all = sum(p.num_envs for p in parts)
    actions = torch.rand((T_LAUNCH, n_all, 4), device='cuda', generator=g) * 2 - 1

    ref = _run(full, actions[:, :n])
    got, off = [], 0
    for p in parts:
        got.append(_run(p, actions[:, off:off + p.num_envs]))
        off += p.num_envs
    finished = 0
    for k in range(LAUNCHES):
        for key, r in ref[k].items():
            cat = torch.cat([g_[k][key] for g_ in got], dim=1)[:, :n]
            assert torch.equal(r, cat), (key, k)
        finished += int((ref[k]['terminated'] | ref[k]['truncated']).sum())
    if n >= 447 and cfg != 'takeoff_simple':                 # U(-1,1) actions end ~10 % of Hover / Circle episodes a step
        assert finished > 0

    planes, pool, pend = _words(full)
    cat = [_words(p) for p in parts]
    assert torch.equal(planes, torch.cat([c[0] for c in cat], dim=1)[:, :n])
    pool_p = torch.cat([c[1] for c in cat], dim=1)[:, :n]
    pend_p = torch.cat([c[2] for c in cat])[:n]
    for s in range(4):
        taken = (((pend | pend_p) >> s) & 1) == 0            # slot s holds a fresh package in both runs
        assert torch.equal(pool[s][taken], pool_p[s][taken]), s

    if n_all == n:
        st = full.episode_stats().cpu()
        sp = [p.episode_stats().cpu() for p in parts]
        assert st[0] == sum(s[0] for s in sp) and st[3] == sum(s[3] for s in sp)
        assert st[4] == min(s[4] for s in sp) and st[6] == min(s[6] for s in sp)
        assert st[5] == max(s[5] for s in sp) and st[7] == max(s[7] for s in sp)
        for k in (1, 2):                                     # float64 sums grouped by block: rounding order only
            assert abs(float(st[k]) - float(sum(s[k] for s in sp))) <= 1e-12 * max(1.0, abs(float(st[k])))
