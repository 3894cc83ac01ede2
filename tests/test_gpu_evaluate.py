"""pdx_evaluate / policy_io.evaluate_many: P policies x E shared episodes in one launch.

  * decomposition: every recorded action is the CUDA-core policy kernel's mean on the recorded observation (bit
    for bit), replaying the recorded actions through VecEnv.step reproduces the recorded observations, rewards,
    costs and flags (same step body, other instantiation: 4e-6 x (1 + |value|), flags equal), and the returned
    returns / lengths / costs are exactly the alive-masked float64 sums of the records;
  * shared episodes: a policy's results do not depend on the other policies of the call;
  * the reference's exported policies run in all three control modes."""
import glob
import os

import numpy as np
import pytest
import torch

from phoenix_drone_simulation_b200 import VecEnv
from phoenix_drone_simulation_b200.lib import PhoenixB200Error
from phoenix_drone_simulation_b200.policy_io import _evaluate_many, evaluate_many, load_policy_json
from phoenix_drone_simulation_b200.rollout import ActorCritic

pytestmark = pytest.mark.gpu
KAT_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden_collector', 'kat_models')


def _policies(P, obs_dim, hidden=(50, 50), stdz=True, seed=0):
    out = []
    for k in range(P):
        torch.manual_seed(1000 * seed + k)
        ac = ActorCritic(obs_dim, pi_hidden=hidden, use_standardized_obs=stdz, policy_kernel='cuda')
        with torch.no_grad():
            if stdz:
                ac.obs_oms.mean.copy_(torch.randn(obs_dim, device='cuda') * 0.1)
                ac.obs_oms.std.copy_(torch.rand(obs_dim, device='cuda') * 0.5 + 0.75)
            for m in ac.pi:
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
        out.append(ac)
    return out


def _check_decomposition(env_id, policies, E, seed, exact_policy=True, tol=4e-6, **kw):
    """exact_policy=False: observations wider than the stand-alone policy kernel's shared-memory plan (its critic
    and 256 hidden columns do not fit next to a 384-wide actor); the actions are then checked against the torch
    actor in float32 (1e-5)."""
    ret, length, cost, rec = _evaluate_many(env_id, policies, E, seed, 'cuda', True, kw)
    P = len(policies)
    T = rec['obs'].shape[0]
    assert ret.shape == cost.shape == length.shape == (P, E) and length.dtype == np.int64
    assert ((length >= 1) & (length <= T)).all() and np.isfinite(ret).all() and np.isfinite(cost).all()
    L = torch.as_tensor(length, device='cuda')
    twin = VecEnv(env_id, E, seed=seed, auto_reset=False, **kw)
    o0 = twin.reset().clone()
    rel = lambda x, y: float(((x - y).abs() / (1.0 + y.abs())).max()) if x.numel() else 0.0
    worst, n_term, n_trunc = {'obs': 0.0, 'reward': 0.0, 'cost': 0.0}, 0, 0
    act = torch.empty((E, 4), device='cuda'); val = torch.empty(E, device='cuda'); lp = torch.empty(E, device='cuda')
    mu = torch.empty((E, 4), device='cuda')
    for p, ac in enumerate(policies):
        assert torch.equal(rec['obs'][0, p], o0), p                                   # (a)
        env = VecEnv(env_id, E, seed=seed, auto_reset=False, **kw)
        env.reset()
        ret_ref = torch.zeros(E, dtype=torch.float64, device='cuda')
        cost_ref = torch.zeros(E, dtype=torch.float64, device='cuda')
        len_ref = torch.zeros(E, dtype=torch.int64, device='cuda')
        alive = torch.ones(E, dtype=torch.bool, device='cuda')
        for t in range(int(L[p].max())):
            done = torch.isnan(rec['act'][t, p, :, 0])          # not recorded: the episode's block had stopped
            assert not bool((done & alive).any()), (p, t)
            if exact_policy:
                ac._launch_into(rec['obs'][t, p].nan_to_num().contiguous(), act, val, lp, mu, counter=0)
                assert torch.equal(mu[~done], rec['act'][t, p][~done]), (p, t)        # (b)
            else:
                o_t = rec['obs'][t, p][~done]
                ref = ac.pi(ac.obs_oms(o_t) if ac.obs_oms else o_t).detach()
                torch.testing.assert_close(rec['act'][t, p][~done], ref, rtol=1e-5, atol=1e-5)
            o, r, te, tr, info = env.step(rec['act'][t, p].nan_to_num().contiguous())
            a = alive
            assert torch.equal(te[a], rec['terminated'][t, p][a].bool()), (p, t)      # (c)
            assert torch.equal(tr[a], rec['truncated'][t, p][a].bool()), (p, t)
            worst['reward'] = max(worst['reward'], rel(rec['reward'][t, p][a], r[a]))
            worst['cost'] = max(worst['cost'], rel(rec['cost'][t, p][a], info['cost'][a]))
            nxt = a & (L[p] > t + 1)
            if t + 1 < T:
                worst['obs'] = max(worst['obs'], rel(rec['obs'][t + 1, p][nxt], o[nxt]))
            ret_ref += torch.where(a, rec['reward'][t, p].double(), torch.zeros_like(ret_ref))   # (d)
            cost_ref += torch.where(a, rec['cost'][t, p].double(), torch.zeros_like(cost_ref))
            len_ref += a
            end = a & (rec['terminated'][t, p].bool() | rec['truncated'][t, p].bool())
            n_term += int((a & rec['terminated'][t, p].bool()).sum()); n_trunc += int((end & ~rec['terminated'][t, p].bool()).sum())
            alive = a & ~end
        assert not bool(alive.any())
        assert torch.equal(len_ref, L[p]), p
        assert torch.equal(ret_ref, torch.as_tensor(ret[p], device='cuda')), p
        assert torch.equal(cost_ref, torch.as_tensor(cost[p], device='cuda')), p
    assert max(worst.values()) <= tol, worst
    print(f'{env_id} {kw}: P={P} E={E}: in-kernel step vs VecEnv.step {worst}, {n_term} terminated, '
          f'{n_trunc} truncated, mean length {length.mean():.1f}')
    return n_term, n_trunc


CONFIGS = [
    # id, env_id, env kwargs, P, E, pi_hidden, standardised
    ('hover_simple', 'DroneHoverSimpleEnv-v0', dict(max_episode_steps=30), 3, 100, (50, 50), True),
    ('hover_bullet', 'DroneHoverBulletEnv-v0', dict(max_episode_steps=25), 1, 128, (50, 50), True),
    ('circle_simple_h8', 'DroneCircleSimpleEnv-v0', dict(max_episode_steps=20, observation_history_size=8), 3, 1, (64, 64), True),
    ('takeoff_bullet', 'DroneTakeOffBulletEnv-v0', dict(max_episode_steps=20), 37, 128, (50, 50), True),
    ('hover_no_noise', 'DroneHoverSimpleEnv-v0', dict(max_episode_steps=40, observation_noise=0), 3, 300, (10, 10), True),
    ('no_standardisation', 'DroneHoverSimpleEnv-v0', dict(max_episode_steps=30), 3, 128, (50, 50), False),
    ('circle_bullet_attrate', 'DroneCircleBulletEnv-v0', dict(max_episode_steps=30, control_mode='AttitudeRate',
                                                            aggregate_phy_steps=4), 2, 100, (64, 64), True),
    ('takeoff_simple_h16', 'DroneTakeOffSimpleEnv-v0', dict(max_episode_steps=20, observation_history_size=16), 2, 64,
     (64, 64), True),
]


@pytest.mark.parametrize('name,env_id,kw,P,E,hidden,stdz', CONFIGS, ids=[c[0] for c in CONFIGS])
def test_evaluate_kernel_is_policy_kernel_plus_env_kernel(name, env_id, kw, P, E, hidden, stdz):
    obs_dim = VecEnv(env_id, 1, **kw).obs_dim
    _check_decomposition(env_id, _policies(P, obs_dim, hidden, stdz, seed=len(name)), E, seed=7,
                         exact_policy=obs_dim <= 192, **kw)


def test_terminations_and_truncations_both_occur():
    n_term, n_trunc = _check_decomposition('DroneHoverSimpleEnv-v0', _policies(4, 34, seed=3), 200, seed=11,
                                           max_episode_steps=30)
    assert n_term > 0 and n_trunc > 0, (n_term, n_trunc)


@pytest.mark.parametrize('env_id', ['DroneCircleBulletEnv-v0', 'DroneHoverSimpleEnv-v0'])
def test_results_of_a_policy_do_not_depend_on_the_other_policies(env_id):
    obs_dim = VecEnv(env_id, 1).obs_dim
    A, B, Cp = _policies(3, obs_dim, seed=5)
    alone = evaluate_many(env_id, [A], 128, seed=3)
    abc = evaluate_many(env_id, [A, B, Cp], 128, seed=3)
    ca = evaluate_many(env_id, [Cp, A], 128, seed=3)
    for k in range(3):
        assert np.array_equal(alone[k][0], abc[k][0]) and np.array_equal(alone[k][0], ca[k][1]), k
        assert np.array_equal(abc[k][2], ca[k][0]), k
    twice = evaluate_many(env_id, [A, A], 128, seed=3)
    for k in range(3):
        assert np.array_equal(twice[k][0], twice[k][1]) and np.array_equal(twice[k][0], alone[k][0]), k
    assert alone[1].max() > 1


def _kat_by_mode():
    groups = {}
    for f in sorted(glob.glob(os.path.join(KAT_DIR, '*_model.json'))):
        groups.setdefault(os.path.basename(f).split('_seed_')[0], []).append(f)
    return groups


@pytest.mark.parametrize('mode,agg', [('PWM', 2), ('AttitudeRate', 4), ('Attitude', 8)])
def test_reference_exported_policies(mode, agg):
    files = _kat_by_mode()[mode]
    assert len(files) == 2
    pols = [load_policy_json(f, policy_kernel='cuda') for f in files]
    kw = dict(control_mode=mode, aggregate_phy_steps=agg)
    # Attitude control runs the two-level PID cascade on each of 8 sub-steps: there the two float32 instantiations of
    # the step body differ by up to 5.2e-6 x (1 + |value|) in an observation entry (measured on a B200), already
    # within the first 10 steps -- a per-step rounding difference, not a drift (flags and rewards stay equal / 1e-7)
    _check_decomposition('DroneCircleBulletEnv-v0', pols, 128, seed=1, max_episode_steps=10,
                         tol=1e-5 if mode == 'Attitude' else 4e-6, **kw)
    ret, length, cost = evaluate_many('DroneCircleBulletEnv-v0', pols, 128, seed=1, **kw)
    assert np.isfinite(ret).all() and np.isfinite(cost).all()
    assert ((length >= 1) & (length <= 500)).all()
    print(f'{mode}: mean return {ret.mean(1)}, mean length {length.mean(1)}')


def test_mixed_policy_sets_and_unsupported_engines_are_rejected():
    with pytest.raises(ValueError):
        evaluate_many('DroneHoverSimpleEnv-v0', _policies(1, 34) + _policies(1, 34, hidden=(64, 64)), 8)
    with pytest.raises(ValueError):
        evaluate_many('DroneHoverSimpleEnv-v0', _policies(1, 34) + _policies(1, 34, stdz=False), 8)
    with pytest.raises(PhoenixB200Error):
        evaluate_many('DroneHoverSimpleEnv-v0', _policies(2, 34), 8, dtype=torch.float64)
    with pytest.raises(PhoenixB200Error):
        evaluate_many('DroneHoverSimpleEnv-v0', _policies(2, 34), 8, rng='tape')
