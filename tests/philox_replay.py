"""Shared harness of the Philox step-kernel tests: one configuration of the production step kernel (k_rollout with the
pooled reset packages) run three ways and replayed through the float64 oracle.

`replay_case` runs N environments for T steps with a time limit and checks:
  * single-step launches against one fused step_many launch: bit for bit;
  * the dump instantiation (pdx_dump_draws: the same draws, the reset done by the owning thread instead of a
    package): flags equal, values within DUMP_TOL;
  * the float64 CPU oracle, built from the same keyword arguments, replaying the dumped draws on every 7th
    environment: within ORACLE_TOL;
  * episode_counters() moved by exactly the number of episodes each environment finished.
"""
import numpy as np
import torch

# production vs dump instantiation.  float64: no FMA contraction in either (-fmad=false), the only difference is that
# a package enters the carried gyro words by linear superposition (test_philox_path_equals_tape_semantics).  float32:
# 4e-6 x (1 + |value|), the bound of test_float32_production_kernel_matches_dump_and_oracle (two instantiations may
# contract differently in the last bit, plus one more rounding through the superposition; episodes here last <= 8
# steps, so nothing accumulates).
DUMP_TOL = {torch.float64: 1e-12, torch.float32: 4e-6}
# engine vs float64 oracle on the dumped draws: test_gpu_parity's F64_TOL and F32_TOL
ORACLE_TOL = {torch.float64: 1e-9, torch.float32: 5e-4}


def vec(*a, **k):
    from phoenix_drone_simulation_b200 import VecEnv
    return VecEnv(*a, **k)


def err(x, y, dtype):
    """float64: max |x - y|; float32: max |x - y| / (1 + |y|) (rewards reach -100)."""
    if x.numel() == 0:
        return 0.0
    d = (x.double() - y.double()).abs()
    if dtype == torch.float32:
        d = d / (1.0 + y.double().abs())
    return float(d.max())


def actions(env, T, N, seed):
    """Hover / Circle: U(-1,1).  TakeOff never terminates: the hover action + 0.3 N(0,1)."""
    rng = np.random.default_rng(seed)
    if 'TakeOff' in env.env_id:
        a = env.cfg.hover_action + 0.3 * rng.standard_normal((T, N, 4))
    else:
        a = rng.uniform(-1.0, 1.0, (T, N, 4))
    return torch.as_tensor(a.astype(np.float32), device='cuda')


def outs(T, N, D, dtype):
    z = lambda *s, dt=dtype: torch.zeros(s, dtype=dt, device='cuda')
    return {'obs': z(T, N, D), 'reward': z(T, N), 'cost': z(T, N), 'terminated': z(T, N, dt=torch.uint8),
            'truncated': z(T, N, dt=torch.uint8), 'final_obs': z(T, N, D)}


def replay_case(env_id, dtype, kw, N, T, max_steps, seed):
    """`kw`: EnvConfig keyword arguments, given unchanged to the VecEnvs and to the OracleEnv (max_episode_steps =
    `max_steps` goes to the VecEnvs only: the oracle has no time limit, the replay applies it).  Returns (production
    vs dump, engine vs oracle, episodes ended) after asserting them."""
    from oracle.phoenix_oracle import OracleEnv, TapeSource
    mk = lambda: vec(env_id, N, dtype=dtype, seed=seed, keep_final_obs=True, max_episode_steps=max_steps, **kw)
    dump, single, fused = mk(), mk(), mk()
    init_tape = dump.dump_init().cpu().numpy()
    obs0, rt = dump.dump_reset()
    obs0 = obs0.double().cpu().numpy().copy()
    err_dump = err(single.reset(), dump.obs, dtype)
    assert torch.equal(fused.reset(), single.obs)
    acts = actions(single, T, N, seed)
    out = outs(T, N, single.obs_dim, dtype)
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
        err_dump = max(err_dump, err(o, dump.obs, dtype), err(r, dump.reward, dtype), err(info['cost'], dump.cost, dtype),
                       err(single.final_obs[fin], dump.final_obs[fin], dtype))
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
        o = OracleEnv(env_id, TapeSource(reset_tapes[c], step_tapes[c], init_tape[:, c]), **kw)
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
    label = ' '.join(f'{k}={v}' for k, v in kw.items())
    print(f'{env_id} {label} {dtype}: production vs dump {err_dump:.2e}, vs oracle {worst:.2e}, '
          f'{int(n_fin.sum())} episodes ended')
    assert worst <= ORACLE_TOL[dtype], worst
    return err_dump, worst, int(n_fin.sum())
