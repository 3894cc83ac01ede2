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
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

EP_PERIOD = 1 << 28
# production vs dump instantiation.  float64: no FMA contraction in either (-fmad=false), the only difference is that
# a package enters the carried gyro words by linear superposition (test_philox_path_equals_tape_semantics).  float32:
# 4e-6 x (1 + |value|), the bound of test_float32_production_kernel_matches_dump_and_oracle (two instantiations may
# contract differently in the last bit, plus one more rounding through the superposition; episodes here last <= 8
# steps, so nothing accumulates).
DUMP_TOL = {torch.float64: 1e-12, torch.float32: 4e-6}
# engine vs float64 oracle on the dumped draws: test_gpu_parity's F64_TOL and F32_TOL
ORACLE_TOL = {torch.float64: 1e-9, torch.float32: 5e-4}

IDS = ['DroneHoverSimpleEnv-v0', 'DroneHoverBulletEnv-v0', 'DroneCircleSimpleEnv-v0', 'DroneCircleBulletEnv-v0',
       'DroneTakeOffSimpleEnv-v0', 'DroneTakeOffBulletEnv-v0']
CASES = [(env_id, noise, ctrl, dtype)
         for k, env_id in enumerate(IDS) for noise in (1, 0) for ctrl in ('PWM', ('AttitudeRate', 'Attitude')[k % 2])
         for dtype in (torch.float32, torch.float64)]


def _vec(*a, **k):
    from phoenix_drone_simulation_b200 import VecEnv
    return VecEnv(*a, **k)


def _err(x, y, dtype):
    """float64: max |x - y|; float32: max |x - y| / (1 + |y|) (rewards reach -100)."""
    if x.numel() == 0:
        return 0.0
    d = (x.double() - y.double()).abs()
    if dtype == torch.float32:
        d = d / (1.0 + y.double().abs())
    return float(d.max())


def _actions(env, T, N, seed):
    """Hover / Circle: U(-1,1).  TakeOff never terminates: the hover action + 0.3 N(0,1)."""
    rng = np.random.default_rng(seed)
    if 'TakeOff' in env.env_id:
        a = env.cfg.hover_action + 0.3 * rng.standard_normal((T, N, 4))
    else:
        a = rng.uniform(-1.0, 1.0, (T, N, 4))
    return torch.as_tensor(a.astype(np.float32), device='cuda')


def _outs(T, N, D, dtype):
    z = lambda *s, dt=dtype: torch.zeros(s, dtype=dt, device='cuda')
    return {'obs': z(T, N, D), 'reward': z(T, N), 'cost': z(T, N), 'terminated': z(T, N, dt=torch.uint8),
            'truncated': z(T, N, dt=torch.uint8), 'final_obs': z(T, N, D)}


@pytest.mark.parametrize('env_id,noise,ctrl,dtype', CASES)
def test_philox_step_matches_dump_and_oracle(env_id, noise, ctrl, dtype):
    """N = 100 environments (three full warps and a ragged one), T = 40 steps, time limit 8 steps (TakeOff 6):
    U(-1,1) actions alone end 0 to 5 episodes per environment in 40 steps (oracle, per id and control mode;
    AttitudeRate Hover none), so the time limit is what keeps the package pool busy.  Asserts flags equal between
    all four, the bounds above, and that episode_counters() moved by exactly the number of episodes each
    environment finished.  Largest values seen on a B200 (37 of the 48 cases printed): production vs dump 2.0e-7
    (float32) and 8.9e-16 (float64); float32 vs oracle 1.9e-4 (Hover-Simple, noise off, AttitudeRate), float64 vs
    oracle 3.7e-10."""
    from oracle.phoenix_oracle import OracleEnv, TapeSource
    N, T = 100, 40
    max_steps = 6 if 'TakeOff' in env_id else 8
    kw = dict(observation_noise=noise, control_mode=ctrl, max_episode_steps=max_steps)
    seed = 1000 + CASES.index((env_id, noise, ctrl, dtype))
    mk = lambda: _vec(env_id, N, dtype=dtype, seed=seed, keep_final_obs=True, **kw)
    dump, single, fused = mk(), mk(), mk()
    init_tape = dump.dump_init().cpu().numpy()
    obs0, rt = dump.dump_reset()
    obs0 = obs0.double().cpu().numpy().copy()
    err_dump = _err(single.reset(), dump.obs, dtype)
    assert torch.equal(fused.reset(), single.obs)
    acts = _actions(single, T, N, seed)
    out = _outs(T, N, single.obs_dim, dtype)
    fused.step_many(acts, out)

    cols = list(range(0, N, 7))
    reset_tapes = {c: [rt[:, c].cpu().numpy().copy()] for c in cols}
    step_tapes = {c: [] for c in cols}
    rec = []
    n_fin = torch.zeros(N, dtype=torch.int64, device='cuda')
    n_trunc = torch.zeros(N, dtype=torch.int64, device='cuda')
    for t in range(T):
        ts, tr = dump.dump_step(acts[t])
        o, r, te, tu, info = single.step(acts[t])
        fin = te | tu
        assert torch.equal(te, dump.terminated) and torch.equal(tu, dump.truncated), t
        # one fused launch == single-step launches of the same instantiation
        assert torch.equal(out['obs'][t], o) and torch.equal(out['reward'][t], r) and torch.equal(out['cost'][t], info['cost']), t
        assert torch.equal(out['terminated'][t].bool(), te) and torch.equal(out['truncated'][t].bool(), tu), t
        assert torch.equal(out['final_obs'][t][fin], single.final_obs[fin]), t
        err_dump = max(err_dump, _err(o, dump.obs, dtype), _err(r, dump.reward, dtype), _err(info['cost'], dump.cost, dtype),
                       _err(single.final_obs[fin], dump.final_obs[fin], dtype))
        n_fin += fin.long()
        n_trunc += tu.long()
        f = fin[cols].cpu().numpy()
        rec.append((dump.obs[cols].double().cpu().numpy(), dump.reward[cols].double().cpu().numpy(),
                    dump.terminated[cols].cpu().numpy(), dump.final_obs[cols].double().cpu().numpy(), f))
        ts, tr = ts[:, cols].cpu().numpy(), tr[:, cols].cpu().numpy()
        for j, c in enumerate(cols):
            step_tapes[c].append(ts[:, j].copy())
            if f[j]:
                reset_tapes[c].append(tr[:, j].copy())
    assert torch.equal(single.state, fused.state)
    assert err_dump <= DUMP_TOL[dtype], err_dump
    # reset traffic: every environment finishes at least T // max_steps episodes (TakeOff: all of them truncations)
    assert int(n_fin.sum()) >= 2 * N and bool((n_fin >= T // max_steps).all())
    assert 'TakeOff' not in env_id or torch.equal(n_trunc, n_fin)
    for e in (single, fused, dump):
        assert torch.equal(e.episode_counters()[0], n_fin)

    worst = 0.0
    for j, c in enumerate(cols):
        o = OracleEnv(env_id, TapeSource(reset_tapes[c], step_tapes[c], init_tape[:, c]),
                      observation_noise=noise, control_mode=ctrl)
        ob, _ = o.reset()
        worst = max(worst, float(np.max(np.abs(ob - obs0[c]))))
        n_ep = 0
        for t in range(T):
            ob, r, term, _, _ = o.step(acts[t, c].cpu().numpy())
            n_ep += 1
            obs_g, rew_g, term_g, fin_obs_g, fin = rec[t]
            assert bool(term_g[j]) == bool(term), (c, t)
            assert bool(fin[j]) == (term or n_ep == max_steps), (c, t)
            got = fin_obs_g[j] if fin[j] else obs_g[j]
            worst = max(worst, float(np.max(np.abs(got - ob))), abs(float(rew_g[j]) - r))
            if fin[j]:
                ob, _ = o.reset()
                n_ep = 0
                worst = max(worst, float(np.max(np.abs(obs_g[j] - ob))))
    print(f'{env_id} noise={noise} {ctrl} {dtype}: production vs dump {err_dump:.2e}, vs oracle {worst:.2e}, '
          f'{int(n_fin.sum())} episodes ended')
    assert worst <= ORACLE_TOL[dtype], worst


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
