"""The production Philox step kernels -- k_rollout with the pooled reset packages -- pinned for every instantiation,
and the auto-reset counter that keys the packages pinned across the ranges where its encoding could break.

(a) Every Philox step instantiation (dtype x task x physics x noise x PWM / PID; the two PID modes share one
    instantiation, so AttitudeRate and Attitude alternate across the env ids) against:
      * one fused step_many launch: bit for bit;
      * the dump instantiation (pdx_dump_draws: the same draws, the reset done by the owning thread instead of a
        package): flags equal, values within DUMP_TOL;
      * the float64 CPU oracle replaying the dumped draws on every 7th environment: within ORACLE_TOL.
(b) The ep_index word ((e << 4) | pending bits, e = auto-resets consumed modulo 2^28) started just below 2^19,
    2^20, 2^27 and 2^28.  float32 holds the word's bit pattern, so these are the points where that pattern turns
    from denormal to normal, where a float VALUE of 16 e + pend would stop being exact, where the pattern becomes
    a NaN / negative pattern (and a float64 value would overflow an int), and the wrap of e.
"""
import pytest
import torch

from philox_replay import DUMP_TOL, replay_case
from philox_replay import actions as _actions, err as _err, vec as _vec

pytestmark = pytest.mark.gpu

EP_PERIOD = 1 << 28

IDS = ['DroneHoverSimpleEnv-v0', 'DroneHoverBulletEnv-v0', 'DroneCircleSimpleEnv-v0', 'DroneCircleBulletEnv-v0',
       'DroneTakeOffSimpleEnv-v0', 'DroneTakeOffBulletEnv-v0']
CASES = [(env_id, noise, ctrl, dtype)
         for k, env_id in enumerate(IDS) for noise in (1, 0) for ctrl in ('PWM', ('AttitudeRate', 'Attitude')[k % 2])
         for dtype in (torch.float32, torch.float64)]


@pytest.mark.parametrize('env_id,noise,ctrl,dtype', CASES)
def test_philox_step_matches_dump_and_oracle(env_id, noise, ctrl, dtype):
    """N = 100 environments (three full warps and a ragged one), T = 40 steps, time limit 8 steps (TakeOff 6):
    U(-1,1) actions alone end 0 to 5 episodes per environment in 40 steps (oracle, per id and control mode;
    AttitudeRate Hover none), so the time limit is what keeps the package pool busy.  Asserts flags equal between
    all four, the bounds above, and that episode_counters() moved by exactly the number of episodes each
    environment finished.  Largest values seen on a B200 (37 of the 48 cases printed): production vs dump 2.0e-7
    (float32) and 8.9e-16 (float64); float32 vs oracle 1.9e-4 (Hover-Simple, noise off, AttitudeRate), float64 vs
    oracle 3.7e-10."""
    max_steps = 6 if 'TakeOff' in env_id else 8
    replay_case(env_id, dtype, dict(observation_noise=noise, control_mode=ctrl), N=100, T=40, max_steps=max_steps,
                seed=1000 + CASES.index((env_id, noise, ctrl, dtype)))


EDGES = [(1 << 19) - 3,    # float32 bit pattern: denormal -> normal
         (1 << 20) - 3,    # a float32 VALUE 16 e + pend stops being exact
         (1 << 27) - 3,    # float32 pattern -> NaN / negative patterns; 16 e overflows an int
         (1 << 28) - 3]    # e wraps


def _start_at(env, dump, e0, N):
    """reset, counters -> (e0, all four slots pending), one hover step: no episode ends, so no package is taken
    before the flush at the end of the step has rebuilt each environment's next one under its new key."""
    for e in (env, dump):
        e.set_episode_counters(e0, 0b1111)
        ep, pend = e.episode_counters()
        assert bool((ep == e0).all()) and bool((pend == 15).all())
    hover = torch.full((N, 4), env.cfg.hover_action, dtype=torch.float32, device='cuda')
    _, _, te, tu, _ = env.step(hover)
    dump.dump_step(hover)
    assert not bool((te | tu).any()) and not bool((dump.terminated | dump.truncated).any())
    ep, pend = env.episode_counters()
    assert bool((ep == e0).all()) and not bool(((pend >> ((e0 + 1) % 4)) & 1).any())
    return _err(env.obs, dump.obs, env.dtype)


@pytest.mark.parametrize('e0', EDGES)
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('env_id', ['DroneHoverBulletEnv-v0', 'DroneCircleSimpleEnv-v0'])
def test_episode_counter_edges(env_id, dtype, e0):
    """4,096 environments, T = 32 steps (one hover step, then U(-1,1)), 2-step time limit: every environment takes
    at least 16 packages past e0, so a pending bit lost early is taken stale within the run.  Production single
    steps against the dump instantiation (its reset keys come from its own word, which never holds pending bits);
    the counter must end at (e0 + finished) mod 2^28 in both.  With a float32 VALUE 16 e + pend in the word, the
    cases from 2^20 - 3 on fail here."""
    N, T = 4096, 32
    mk = lambda: _vec(env_id, N, dtype=dtype, seed=31, keep_final_obs=True, max_episode_steps=2)
    env, dump = mk(), mk()
    err = _err(env.reset(), dump.dump_reset()[0], dtype)
    err = max(err, _start_at(env, dump, e0, N))
    acts = _actions(env, T, N, 7)
    n_fin = torch.zeros(N, dtype=torch.int64, device='cuda')
    for t in range(1, T):
        dump.dump_step(acts[t])
        o, r, te, tu, info = env.step(acts[t])
        fin = te | tu
        assert torch.equal(te, dump.terminated) and torch.equal(tu, dump.truncated), t
        err = max(err, _err(o, dump.obs, dtype), _err(r, dump.reward, dtype), _err(info['cost'], dump.cost, dtype),
                  _err(env.final_obs[fin], dump.final_obs[fin], dtype))
        n_fin += fin.long()
    print(f'{env_id} {dtype} e0 = {e0}: production vs dump {err:.2e}, {int(n_fin.sum())} episodes ended')
    assert bool((n_fin >= T // 2).all())
    assert err <= DUMP_TOL[dtype], err
    for e in (env, dump):
        assert torch.equal(e.episode_counters()[0], (e0 + n_fin) % EP_PERIOD)


@pytest.mark.parametrize('e0', EDGES)
@pytest.mark.parametrize('env_id', ['DroneHoverBulletEnv-v0', 'DroneCircleSimpleEnv-v0'])
def test_collector_episode_counter_edges(env_id, e0):
    """The fused collector (pdx_collect, split-TF32 policy) steps with the same pool code: one 32-step rollout of
    5,000 environments after the protocol above, its stored actions replayed through the dump instantiation (not
    a production twin: that shares the pool, so it would be wrong in the same way)."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
    N, T = 5000, 32
    mk = lambda: _vec(env_id, N, seed=41, keep_final_obs=True, max_episode_steps=2)
    env, dump = mk(), mk()
    err = _err(env.reset(), dump.dump_reset()[0], torch.float32)
    err = max(err, _start_at(env, dump, e0, N))
    ac = ActorCritic(env.obs_dim, policy_kernel='tc', seed=3)
    col = RolloutCollector(env, ac, T)
    col.collect()                                        # (explicit reset first: it keeps the counters)
    assert col.fused_used, 'pdx_collect was not used'
    err = max(err, _err(col.obs[0], dump.dump_reset()[0], torch.float32))
    n_fin = torch.zeros(N, dtype=torch.int64, device='cuda')
    for t in range(T):
        dump.dump_step(col.act[t])
        assert torch.equal(col.term[t].bool(), dump.terminated) and torch.equal(col.trunc[t].bool(), dump.truncated), t
        err = max(err, _err(col.obs[t + 1], dump.obs, torch.float32), _err(col.rew[t], dump.reward, torch.float32),
                  _err(col.cost[t], dump.cost, torch.float32))
        n_fin += (dump.terminated | dump.truncated).long()
    print(f'{env_id} pdx_collect e0 = {e0}: collector vs dump {err:.2e}, {int(n_fin.sum())} episodes ended')
    assert bool((n_fin >= T // 2).all())
    assert err <= DUMP_TOL[torch.float32], err
    for e in (env, dump):
        assert torch.equal(e.episode_counters()[0], (e0 + n_fin) % EP_PERIOD)
