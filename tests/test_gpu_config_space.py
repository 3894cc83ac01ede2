"""The step kernels at non-default EnvConfig options, against the float64 oracle.

Most options are run-time fields of the device configuration: they steer branches inside reset_env, the reset-package
pool and the sub-step loop that the default settings never take (ring of one sub-step, gyro-only sub-steps, the motor
time-constant clamp, 7 instead of 15 domain-randomisation draws, history row modes, a non-default target, ...).
  * CONFIGS: every row runs the production Philox path in both precisions through tests/philox_replay.py (single
    steps, one fused launch, the dump instantiation and the oracle on the dumped draws);
  * host-driven resets: auto_reset=False (what the gymnasium drop-in and simopt use), and masked reset(mask);
  * pdx_collect rollouts at non-default options, replayed through the dump instantiation;
  * (CPU) the oracle's per-phase draw counts equal pdx_tape_slots for every row: a mismatch would misalign every
    tape the replay reads.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from philox_replay import DUMP_TOL, ORACLE_TOL, actions, err, outs, replay_case, vec

DTYPES = [torch.float32, torch.float64]
DT_IDS = ['f32', 'f64']
HS, HB = 'DroneHoverSimpleEnv-v0', 'DroneHoverBulletEnv-v0'
CS, CB = 'DroneCircleSimpleEnv-v0', 'DroneCircleBulletEnv-v0'
TS, TB = 'DroneTakeOffSimpleEnv-v0', 'DroneTakeOffBulletEnv-v0'
PEN = dict(target_pos=(0.3, -0.2, 1.1), penalty_angle=0.05, penalty_velocity=0.02, penalty_terminal=7)

# (env id, EnvConfig kwargs, time limit: None = 8 steps, 6 for TakeOff)
CONFIGS = [
    # latency and motor model
    (HB, dict(latency=0.005), None),                                   # buf_size 1: ring of one sub-step
    (CB, dict(latency=0.004, control_mode='AttitudeRate'), None),      # ring off by rule, reset still draws 4 words
    (HB, dict(use_latency=False, control_mode='Attitude'), None),
    (TB, dict(use_motor_dynamics=False), None),                        # 7 DR draws on Bullet
    (HB, dict(use_latency=False, use_motor_dynamics=False, control_mode='AttitudeRate'), None),
    (CB, dict(motor_time_constant=0.004), None),                       # every draw below dt: Tm = fmax(draw, dt)
    (CS, dict(motor_thrust_noise=0, control_mode='Attitude'), None),
    # resets
    (HS, dict(enable_reset_distribution=False), None),
    (CB, dict(enable_reset_distribution=False, control_mode='AttitudeRate'), None),
    (TS, dict(enable_reset_distribution=False), None),
    (HB, dict(domain_randomization=-1), None),
    (CS, dict(domain_randomization=0, control_mode='AttitudeRate'), None),    # the `> 0` edge
    (HB, dict(domain_randomization=0.3, control_mode='Attitude'), None),
    # sub-steps
    (HS, dict(aggregate_phy_steps=3), None),
    (CS, dict(aggregate_phy_steps=5), None),
    (TB, dict(aggregate_phy_steps=6), None),
    (HB, dict(aggregate_phy_steps=8, control_mode='AttitudeRate'), None),
    (HB, dict(observation_frequency=50, aggregate_phy_steps=4), None),        # obs_rate 4
    (CS, dict(observation_frequency=50, aggregate_phy_steps=2, control_mode='Attitude'), None),   # obs_rate 2
    (TB, dict(observation_frequency=200, aggregate_phy_steps=3, latency=0.01), None),            # obs_rate 1
    (CB, dict(observation_frequency=200, aggregate_phy_steps=1, latency=0.005, control_mode='AttitudeRate'), None),
    # history (row modes: 0 rows as in the output, 1 rotated walk, 2 padded float32 rows)
    (HB, dict(observation_history_size=1), None),                      # aliasing window H - 1 + n_ep <= H
    (TB, dict(observation_history_size=3, control_mode='Attitude'), None),    # D = 72: mode 0
    (CB, dict(observation_history_size=4), None),                      # D = 80: mode 2 in float32
    (HB, dict(observation_history_size=16, control_mode='AttitudeRate'), None),   # D = 272: mode 1
    (TS, dict(observation_history_size=16), None),                     # D = 384: mode 2, widest row
    # reward and physics
    (HS, dict(PEN), None),
    (HB, dict(PEN, control_mode='AttitudeRate'), None),
    (HB, dict(use_ground_effect=True), None),
    (CS, dict(use_ground_effect=True, control_mode='AttitudeRate'), None),
    (CB, dict(lin_damping=0.2, ang_damping=0), None),
    (HS, dict(), 1),                                                   # every environment takes a package every step
    (CB, dict(control_mode='Attitude'), 1),
]


def _time_limit(env_id, limit):
    return limit if limit is not None else (6 if 'TakeOff' in env_id else 8)


def _id(row):
    env_id, kw, limit = row
    tag = ','.join(f'{k}={v}'.replace(' ', '') for k, v in kw.items()) or 'defaults'
    return f"{env_id.replace('Env-v0', '')}-{tag}" + (f'-limit{limit}' if limit else '')


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('row', CONFIGS, ids=[_id(r) for r in CONFIGS])
def test_config_matches_dump_and_oracle(row, dtype):
    """N = 100 (a ragged warp), T = 40, time limit 8 steps (6 for TakeOff, 1 in the last two rows): the package pool
    stays busy.  Asserts what tests/philox_replay.py asserts; prints the two largest errors."""
    env_id, kw, limit = row
    replay_case(env_id, dtype, kw, N=100, T=40, max_steps=_time_limit(env_id, limit),
                seed=2000 + 2 * CONFIGS.index(row) + (dtype == torch.float64))


def test_oracle_draw_counts_match_tape_slots():
    """For every row: the draws the oracle consumes in one reset and one step (counted by dry-running it) equal the
    tape widths the engine lays out (pdx_tape_slots).  Runs without a GPU."""
    import phoenix_drone_simulation_b200 as pds
    from phoenix_drone_simulation_b200 import lib as L
    from oracle.phoenix_oracle import draws_per_phase
    lib = L.load()
    for env_id, kw, _ in CONFIGS:
        for noise in (1, 0):
            k = dict(kw, observation_noise=noise)
            c = pds.EnvConfig(env_id, **k).to_pdx()
            rs, ss, is_ = C.c_int(), C.c_int(), C.c_int()
            assert lib.pdx_tape_slots(C.byref(c), C.byref(rs), C.byref(ss), C.byref(is_)) == 0
            assert draws_per_phase(env_id, **k) == (rs.value, ss.value), (env_id, k)


# ---------------------------------------------------------------------------------------------------------------------
#  host-driven resets
# ---------------------------------------------------------------------------------------------------------------------
def _host(t):
    return t.double().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('env_id', [HS, HB])
def test_no_auto_reset_steps_on_from_the_terminal_state(env_id, dtype):
    """auto_reset=False: an environment whose episode ended keeps stepping from its terminal state, as the reference
    does when nobody calls reset().  N = 100, T = 40, U(-1,1) actions, time limit 8.  Single steps, one fused launch,
    the dump instantiation and the oracle (no reset after the first) over the whole run; `truncated` stays set after
    the limit, `terminated` follows done(), the episode counters do not move, and every step on which an episode is
    over counts in episode_stats() and episode_length (the VecEnv docstring)."""
    from oracle.phoenix_oracle import OracleEnv, TapeSource
    N, T, limit = 100, 40, 8
    mk = lambda: vec(env_id, N, dtype=dtype, seed=77, max_episode_steps=limit, auto_reset=False)
    dump, single, fused = mk(), mk(), mk()
    init_tape = dump.dump_init().cpu().numpy()
    obs0, rt = dump.dump_reset()
    obs0 = _host(obs0).copy()
    rt = rt.cpu().numpy()
    e_dump = err(single.reset(), dump.obs, dtype)
    fused.reset()
    counters0 = single.episode_counters()
    acts = actions(single, T, N, 5)
    out = outs(T, N, single.obs_dim, dtype)
    del out['final_obs']                                   # (no reset writes one)
    fused.step_many(acts, out)
    single.clear_episode_stats()
    ret = torch.zeros(N, dtype=dtype, device='cuda')
    fin_any = torch.zeros(N, dtype=torch.bool, device='cuda')
    n, lens, rets = 0, [], []
    step_tapes, rec = [], []
    for t in range(T):
        ts, _ = dump.dump_step(acts[t])
        o, r, te, tu, info = single.step(acts[t])
        assert torch.equal(te, dump.terminated) and torch.equal(tu, dump.truncated), t
        assert torch.equal(out['obs'][t], o) and torch.equal(out['reward'][t], r), t
        assert torch.equal(out['terminated'][t].bool(), te) and torch.equal(out['truncated'][t].bool(), tu), t
        assert bool((tu == (t + 1 >= limit)).all()), t
        e_dump = max(e_dump, err(o, dump.obs, dtype), err(r, dump.reward, dtype), err(info['cost'], dump.cost, dtype))
        fin = te | tu
        fin_any |= fin
        ret += r                                           # the kernel's ep_return: a running sum in the engine dtype
        assert torch.equal(info['episode_length'], torch.where(fin, t + 1, 0).to(torch.int32)), t
        assert torch.equal(info['episode_return'], torch.where(fin, ret, torch.zeros_like(ret))), t
        n += int(fin.sum())
        lens += [t + 1] * int(fin.sum())
        rets += _host(ret[fin]).tolist()
        step_tapes.append(ts.cpu().numpy())
        rec.append((_host(dump.obs), _host(dump.reward), dump.terminated.cpu().numpy()))
    assert torch.equal(single.state, fused.state)
    assert e_dump <= DUMP_TOL[dtype], e_dump
    assert bool(fin_any.all())
    for e in (single, fused, dump):
        assert all(torch.equal(x, y) for x, y in zip(e.episode_counters(), counters0))
    s = single.episode_stats().cpu().numpy()
    assert s[0] == n and s[3] == sum(lens) and s[6] == min(lens) and s[7] == T
    np.testing.assert_allclose(s[1], sum(rets), rtol=1e-12, atol=1e-9)
    assert s[4] == min(rets) and s[5] == max(rets)

    worst, n_term = 0.0, 0
    for c in range(0, N, 7):
        o = OracleEnv(env_id, TapeSource([rt[:, c]], [ts[:, c] for ts in step_tapes], init_tape[:, c]))
        ob, _ = o.reset()
        worst = max(worst, float(np.max(np.abs(ob - obs0[c]))))
        for t in range(T):
            ob, r, term, _, _ = o.step(acts[t, c].cpu().numpy())
            obs_g, rew_g, term_g = rec[t]
            assert bool(term_g[c]) == bool(term), (c, t)
            n_term += bool(term)
            worst = max(worst, float(np.max(np.abs(obs_g[c] - ob))), abs(float(rew_g[c]) - r))
    print(f'{env_id} auto_reset=False {dtype}: production vs dump {e_dump:.2e}, vs oracle {worst:.2e}, '
          f'{n_term} terminated steps on the replayed columns')
    assert n_term > 0
    assert worst <= ORACLE_TOL[dtype], worst


def _dump_reset_masked(dump, twin, mask):
    """reset(mask) of the dump instantiation: pdx_dump_draws resets every environment, so it runs on `twin` loaded
    with `dump`'s state and counter; the masked environments are copied back.  The draws of an explicit reset depend
    only on (seed, global index, call counter)."""
    twin.load_state_dict(dump.state_dict())
    obs, rt = twin.dump_reset()
    dump._counter = twin._counter                         # the reset call took one counter
    dump.state[:, mask] = twin.state[:, mask]
    dump.obs[mask] = obs[mask]
    return rt


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('env_id', [HB, CS])
def test_masked_reset_matches_dump_and_oracle(env_id, dtype):
    """auto_reset=False, N = 100, time limit 8.  10 steps of U(-1,1), then reset(mask) with a random mask:
      * unmasked environments: every state quad (package pool and ep_index included) and the observation row
        unchanged bit for bit;
      * masked environments: equal to a dump_reset() of a second VecEnv holding a copy of the pre-reset state at the
        same counter (the stale body rates and the gyro bias come from the copied state);
    then 30 steps of the drop-in loop: step, reset(mask=terminated | truncated) from the host.  The whole run is
    compared with the dump instantiation, and every 7th environment replays the dumped draws through the oracle."""
    from oracle.phoenix_oracle import OracleEnv, TapeSource
    N, T1, T2, limit = 100, 10, 30, 8
    mk = lambda: vec(env_id, N, dtype=dtype, seed=91, max_episode_steps=limit, auto_reset=False)
    prod, dump, twin = mk(), mk(), mk()
    cols = list(range(0, N, 7))
    init_tape = dump.dump_init().cpu().numpy()
    obs0, rt = dump.dump_reset()
    obs0, rt = _host(obs0).copy(), rt.cpu().numpy()
    e_dump = err(prod.reset(), dump.obs, dtype)
    # per replayed column: reset tapes, step tapes and the events ('reset', obs) / ('step', t, obs, reward, flags)
    reset_tapes = {c: [rt[:, c].copy()] for c in cols}
    step_tapes = {c: [] for c in cols}
    events = {c: [('reset', obs0[c])] for c in cols}
    acts = actions(prod, T1 + T2, N, 13)
    rng = np.random.default_rng(3)
    n_resets = 0

    def record_reset(mask, rt):
        m = mask.cpu().numpy()
        rt = rt.cpu().numpy()
        for c in cols:
            if m[c]:
                reset_tapes[c].append(rt[:, c].copy())
                events[c].append(('reset', _host(dump.obs[c])))

    for t in range(T1 + T2):
        ts, _ = dump.dump_step(acts[t])
        o, r, te, tu, info = prod.step(acts[t])
        assert torch.equal(te, dump.terminated) and torch.equal(tu, dump.truncated), t
        e_dump = max(e_dump, err(o, dump.obs, dtype), err(r, dump.reward, dtype), err(info['cost'], dump.cost, dtype))
        ts = ts.cpu().numpy()
        for c in cols:
            step_tapes[c].append(ts[:, c].copy())
            events[c].append(('step', t, _host(dump.obs[c]), float(dump.reward[c]), bool(te[c]), bool(tu[c])))
        if t == T1 - 1:                                    # mid-run: a random mask
            mask = torch.as_tensor(rng.random(N) < 0.5, device='cuda')
            keep = ~mask
            state0, obs_before = prod.state.clone(), prod.obs.clone()
            twin.load_state_dict(prod.state_dict())
            tw_obs, _ = twin.dump_reset()
            prod.reset(mask)
            assert torch.equal(prod.state[:, keep], state0[:, keep]) and torch.equal(prod.obs[keep], obs_before[keep])
            e_mask = max(err(prod.state[:, mask], twin.state[:, mask], dtype), err(prod.obs[mask], tw_obs[mask], dtype))
            assert e_mask <= DUMP_TOL[dtype], e_mask
            e_dump = max(e_dump, e_mask)
        elif t >= T1:                                      # the drop-in loop
            mask = te | tu
            if not bool(mask.any()):
                continue
            prod.reset(mask)
        else:
            continue
        record_reset(mask, _dump_reset_masked(dump, twin, mask))
        n_resets += int(mask.sum())
        e_dump = max(e_dump, err(prod.obs, dump.obs, dtype))
        assert prod._counter == dump._counter
    assert e_dump <= DUMP_TOL[dtype], e_dump

    worst = 0.0
    for c in cols:
        o = OracleEnv(env_id, TapeSource(reset_tapes[c], step_tapes[c], init_tape[:, c]))
        n_ep = 0
        for ev in events[c]:
            if ev[0] == 'reset':
                ob, _ = o.reset()
                n_ep = 0
                worst = max(worst, float(np.max(np.abs(ev[1] - ob))))
                continue
            _, t, obs_g, rew_g, term_g, trunc_g = ev
            ob, r, term, _, _ = o.step(acts[t, c].cpu().numpy())
            n_ep += 1
            assert term_g == bool(term) and trunc_g == (n_ep >= limit), (c, t)
            worst = max(worst, float(np.max(np.abs(obs_g - ob))), abs(rew_g - r))
    print(f'{env_id} reset(mask) {dtype}: production vs dump {e_dump:.2e}, vs oracle {worst:.2e}, '
          f'{n_resets} masked resets')
    assert worst <= ORACLE_TOL[dtype], worst


# ---------------------------------------------------------------------------------------------------------------------
#  the fused collector
# ---------------------------------------------------------------------------------------------------------------------
COLLECT = [
    (HB, dict(aggregate_phy_steps=8, observation_frequency=50)),
    (CB, dict(enable_reset_distribution=False, domain_randomization=0)),
    (HB, dict(observation_history_size=1, latency=0.005)),
]


@pytest.mark.gpu
@pytest.mark.parametrize('env_id,kw', COLLECT, ids=[_id((e, k, None)) for e, k in COLLECT])
def test_collector_non_default_options(env_id, kw):
    """pdx_collect (split-TF32 policy) steps with the same rollout_step: one 32-step rollout of 2,000 environments
    with a time limit of 8, its stored actions replayed through the dump instantiation (flags equal, values within
    DUMP_TOL, counters moved by the finished episodes)."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
    N, T = 2000, 32
    mk = lambda: vec(env_id, N, seed=43, keep_final_obs=True, max_episode_steps=8, **kw)
    env, dump = mk(), mk()
    ac = ActorCritic(env.obs_dim, policy_kernel='tc', seed=3)
    col = RolloutCollector(env, ac, T)
    col.collect()
    assert col.fused_used, 'pdx_collect was not used'
    e = err(col.obs[0], dump.dump_reset()[0], torch.float32)
    n_fin = torch.zeros(N, dtype=torch.int64, device='cuda')
    for t in range(T):
        dump.dump_step(col.act[t])
        assert torch.equal(col.term[t].bool(), dump.terminated) and torch.equal(col.trunc[t].bool(), dump.truncated), t
        e = max(e, err(col.obs[t + 1], dump.obs, torch.float32), err(col.rew[t], dump.reward, torch.float32),
                err(col.cost[t], dump.cost, torch.float32))
        n_fin += (dump.terminated | dump.truncated).long()
    print(f'{env_id} {kw} pdx_collect: collector vs dump {e:.2e}, {int(n_fin.sum())} episodes ended')
    assert bool((n_fin >= T // 8).all())
    assert e <= DUMP_TOL[torch.float32], e
    for x in (env, dump):
        assert torch.equal(x.episode_counters()[0], n_fin)
