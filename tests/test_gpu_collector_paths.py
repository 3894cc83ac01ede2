"""The rollout collector's paths against a float64 reference: continuing episodes and time limits through
pdx_collect (final_obs rows, boot values, done = 2), the alternating-launch fallback (policy kernel, then env
kernel; CUDA graphs of the torch policy for float64 environments) and pdx_collect across the observation
widths and networks its plan accepts.

`check_rollout` checks one collected rollout against
  * the float64 networks (oracle.collector_oracle) on the stored observations, with the Gaussian draw of a
    stand-alone CUDA-core policy launch at the same Philox counter (both kernels share Philox and Box-Muller);
    single TF32 against the model of tests/tf32_reference.py;
  * a twin VecEnv that replays the stored actions with single-step launches from the same state;
  * the truncation bookkeeping (boot, final_obs, done), GAE (oracle.rollout_gae) and the statistics.
"""
import math

import numpy as np
import pytest
import torch

from oracle import collector_oracle as co
import tf32_reference as tfr

pytestmark = pytest.mark.gpu

TOL_F32 = 2e-5              # split TF32 / CUDA-core kernels vs float64: |got - ref| / (1 + |ref|)
TOL_ENV = 4e-6              # pdx_collect's step body vs the single-step kernel (other instantiation)
# Single TF32 in pdx_collect passes X and the layer-1 activations as raw float32 words.  Measured on a B200 (1,000 W)
# with test_single_tf32_reference_model: the actor mean is 1.0e-4 from the model with truncated operands and 4.5e-4
# from the model with rounded ones, so the tensor core truncates.  Largest error over all cases of this file: mean
# 1.4e-4, value 5.4e-5 beyond the tanh.approx bound.  Tolerances: about 4x that.
COLLECT_TF32_CONVERT = 'trunc'
TOL_TF32_MU = 6e-4          # |act - model| / (1 + |model|)
TOL_TF32_V = 2e-4           # the TF32 term of the value bound (tanh.approx of layer 2 comes on top, per row)


def _layers(net):
    return [(m.weight.detach().cpu().numpy().copy(), m.bias.detach().cpu().numpy().copy())
            for m in net if isinstance(m, torch.nn.Linear)]


def snapshot(ac, env):
    """What the collect will read, taken before anything updates it."""
    oms = ac.obs_oms
    return dict(mean=oms.mean.detach().cpu().numpy().copy() if oms is not None else None,
                std=oms.std.detach().cpu().numpy().copy() if oms is not None else None,
                eps=oms.eps if oms is not None else 0.0,
                ret_std=float(ac.ret_oms.std) if ac.ret_oms is not None else None,
                log_std=ac.log_std.detach().cpu().numpy().copy(), pi=_layers(ac.pi), v=_layers(ac.v),
                sd={k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in ac.state_dict().items()},
                c0=ac._counter, env_counter=env._counter, env_state=env.state.clone())


def _rel(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float((np.abs(got - ref) / (1.0 + np.abs(ref))).max()) if got.size else 0.0


def _policy_model(rows, snap, precision, convert):
    """(mu, v, per-row tolerance of mu, per-row tolerance of v) of the kernel that ran at `precision`."""
    if precision == 1:
        mu, v, terms = tfr.forward(rows, snap['mean'], snap['std'], snap['eps'], snap['pi'], snap['v'], convert)
        return mu, v, TOL_TF32_MU * (1 + np.abs(mu)), TOL_TF32_V + tfr.tanh_bound(terms)
    zero = np.zeros((rows.shape[0], snap['log_std'].shape[0]))
    _, v, _, mu = co.actor_critic_step(rows, snap['mean'], snap['std'], snap['pi'], snap['v'], snap['log_std'], zero,
                                       norm_eps=snap['eps'])
    return mu, v, TOL_F32 * (1 + np.abs(mu)), TOL_F32 * (1 + np.abs(v))


def check_rollout(col, data, twin, snap, reset, label=''):
    """Asserts everything a collected rollout must satisfy (see the module docstring); returns the max errors."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic
    env, ac, T = col.env, col.ac, col.T
    N, D = env.num_envs, env.obs_dim
    fused = col.fused_used
    torch_policy = env.dtype == torch.float64              # CUDA graphs of the torch modules, torch's draws
    precision = None if torch_policy else ac.tc_precision
    convert = COLLECT_TF32_CONVERT if fused else 'rna'     # k_policy_tc rounds its operands itself
    out = dict(fused_used=fused, tc_precision=ac.tc_precision, policy=0.0, env=0.0, trunc=0, tf32_mu=0.0, tf32_v=0.0)
    std = np.exp(snap['log_std'].astype(np.float32)).astype(np.float64)
    log_std = snap['log_std'].astype(np.float64)
    obs = col.obs.double().cpu().numpy()
    act, val, logp = (x.double().cpu().numpy() for x in (col.act, col.val, col.logp))

    # ---- 1. policy half, float64 reference
    if not torch_policy:
        draw_ac = ActorCritic(D, pi_hidden=tuple(l[0].shape[0] for l in snap['pi'][:2]),
                              v_hidden=tuple(l[0].shape[0] for l in snap['v'][:2]), seed=ac.seed, policy_kernel='cuda')
        draw_ac.load_state_dict(snap['sd'])
        draw_ac.env_offset = ac.env_offset
        a2 = torch.empty((N, 4), device='cuda'); v2 = torch.empty(N, device='cuda')
        l2 = torch.empty(N, device='cuda'); m2 = torch.empty((N, 4), device='cuda')
    for t in range(T + 1):
        rows = obs[t] if t < T else obs[T]
        mu, v, tol_mu, tol_v = _policy_model(rows, snap, precision or 0, convert)
        if t == T:                                            # the cut is bootstrapped with V(obs[T])
            lv = col.last_val.double().cpu().numpy()
            assert (np.abs(lv - v) <= tol_v).all(), (label, 'last_val', float(np.abs(lv - v).max()))
            break
        if torch_policy:
            assert (np.abs(val[t] - v) <= tol_v).all(), (label, t, float(np.abs(val[t] - v).max()))
            z = (act[t] - mu) / std
            ref_lp = (-0.5 * z * z - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
            np.testing.assert_allclose(logp[t], ref_lp, rtol=0, atol=1e-4, err_msg=label)
            assert abs(z.mean()) < 0.25 and abs(z.std() - 1) < 0.25
            out['policy'] = max(out['policy'], _rel(val[t], v))
            continue
        draw_ac._launch_into(col.obs[t].contiguous(), a2, v2, l2, m2, counter=snap['c0'] + 1 + t)
        draw = (a2.double() - m2.double()).cpu().numpy() / std
        a_ref = mu + std * draw
        lp_ref = (-0.5 * draw * draw - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        e_act, e_val = np.abs(act[t] - a_ref), np.abs(val[t] - v)
        assert (e_act <= tol_mu).all(), (label, t, 'act', float(e_act.max()))
        assert (e_val <= tol_v).all(), (label, t, 'val', float(e_val.max()))
        assert _rel(logp[t], lp_ref) <= TOL_F32, (label, t, 'logp', _rel(logp[t], lp_ref))
        if precision == 1:
            out['tf32_mu'] = max(out['tf32_mu'], float(e_act.max()))
            out['tf32_v'] = max(out['tf32_v'], float((e_val - tfr.tanh_bound(tfr.forward(
                rows, snap['mean'], snap['std'], snap['eps'], snap['pi'], snap['v'], convert)[2])).max()))
        else:
            out['policy'] = max(out['policy'], _rel(act[t], a_ref), _rel(val[t], v))

    # ---- 2. env half: replay the stored actions through the twin from the same state
    twin.state.copy_(snap['env_state'])
    twin._counter = snap['env_counter']
    twin.clear_episode_stats()
    if reset:
        assert torch.equal(twin.reset(), col.obs[0]), label
    term, trunc = col.term.cpu().numpy(), col.trunc.cpu().numpy()
    boot = col.boot.double().cpu().numpy()
    assert (boot[trunc == 0] == 0).all(), (label, 'boot must be 0 without a truncation')
    for t in range(T):
        o, r, te, tr, info = twin.step(col.act[t].contiguous())
        assert torch.equal(te.to(torch.uint8), col.term[t]) and torch.equal(tr.to(torch.uint8), col.trunc[t]), (label, t)
        assert torch.equal(info['cost'], col.cost[t]), (label, t)
        if fused:
            e = max(_rel(col.obs[t + 1].double().cpu().numpy(), o.double().cpu().numpy()),
                    _rel(col.rew[t].double().cpu().numpy(), r.double().cpu().numpy()))
            assert e <= TOL_ENV, (label, t, e)
            out['env'] = max(out['env'], e)
        else:
            assert torch.equal(col.obs[t + 1], o) and torch.equal(col.rew[t], r), (label, t)
        # ---- 3. truncation bookkeeping
        idx = np.nonzero(trunc[t])[0]
        if idx.size:
            final = twin.final_obs[torch.as_tensor(idx, device='cuda')]
            rows = final.double().cpu().numpy()
            _, v, _, tol_v = _policy_model(rows, snap, precision or 0, 'rna')     # ActorCritic.value: k_policy_tc
            assert (np.abs(boot[t, idx] - v) <= tol_v).all(), (label, t, 'boot', float(np.abs(boot[t, idx] - v).max()))
            if fused:
                assert _rel(col._final_obs_T[t][torch.as_tensor(idx, device='cuda')].double().cpu().numpy(), rows) <= TOL_ENV, (label, t)
            out['trunc'] += int(idx.size)
    done = data['done'].cpu().numpy()
    np.testing.assert_array_equal(done, np.where(trunc > 0, 2, np.where(term > 0, 1, 0)), err_msg=label)
    if fused:                                              # the state written back at the end of the pass
        for name in ('xyz', 'vel', 'ou', 'last_action', 'ep_length', 'gyro_bias', 'gyro_lpf', 'dt', 'mass'):
            torch.testing.assert_close(env.get_state(name), twin.get_state(name), rtol=1e-5, atol=1e-5)
    else:
        assert torch.equal(env.state, twin.state), label

    # ---- 4. GAE on whole columns: first, last, truncated ones, one with a termination
    cols = {0, N - 1}
    cols.update(int(i) for i in np.nonzero(trunc.any(0))[0][:48])
    cols.update(int(i) for i in np.nonzero(term.any(0))[0][:8])
    cols = sorted(cols)
    rew = col.rew.double().cpu().numpy()
    a0, t0, d0 = co.rollout_gae(rew[:, cols], val[:, cols], done[:, cols], boot[:, cols],
                                col.last_val.double().cpu().numpy()[cols], col.gamma, col.lam, snap['ret_std'])
    for k, ref in (('adv', a0), ('target_v', t0), ('discounted_ret', d0)):
        np.testing.assert_allclose(data[k].cpu().numpy()[:, cols], ref, rtol=2e-4, atol=2e-4, err_msg=f'{label} {k}')

    # ---- 5. statistics
    got, ref = data['episode_stats']._stats.cpu().numpy(), twin.episode_stats().cpu().numpy()
    assert got[0] == ref[0] == int((done != 0).sum()), label
    assert got[3] == ref[3] and got[6] == ref[6] and got[7] == ref[7], label      # lengths
    if got[0]:
        if fused:                                          # returns of rewards that agree to TOL_ENV per step
            len_max = float(ref[7])
            np.testing.assert_allclose(got[[1, 2]], ref[[1, 2]], rtol=TOL_ENV * len_max * 4, err_msg=label)
            np.testing.assert_allclose(got[[4, 5]], ref[[4, 5]], rtol=0, atol=TOL_ENV * len_max * (1 + np.abs(ref[[4, 5]])).max(), err_msg=label)
        else:
            np.testing.assert_allclose(got[[1, 2]], ref[[1, 2]], rtol=1e-6, err_msg=label)
            np.testing.assert_array_equal(got[[4, 5]], ref[[4, 5]], err_msg=label)
    if fused and ac.obs_oms is not None:
        mom, shift = data['obs_moments']
        x = col.obs[:T].reshape(T * N, -1).double() - shift.double()
        torch.testing.assert_close(mom[:D], x.sum(0), rtol=1e-6, atol=1e-3)
        torch.testing.assert_close(mom[D:], (x * x).sum(0), rtol=1e-6, atol=1e-3)
    return out


def _make(env_id, kernel, N, T, reset_each, seed=21, env_offset=640, pi_hidden=(50, 50), v_hidden=(64, 64),
          dtype=torch.float32, **env_kw):
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
    env = VecEnv(env_id, N, seed=seed, keep_final_obs=True, env_offset=env_offset, dtype=dtype, **env_kw)
    twin = VecEnv(env_id, N, seed=seed, keep_final_obs=True, env_offset=env_offset, dtype=dtype, **env_kw)
    ac = ActorCritic(env.obs_dim, pi_hidden=pi_hidden, v_hidden=v_hidden, policy_kernel=kernel, seed=5)
    with torch.no_grad():
        ac.obs_oms.mean.copy_(torch.randn(env.obs_dim, device='cuda') * 0.1)
        ac.obs_oms.std.copy_(torch.rand(env.obs_dim, device='cuda') * 0.5 + 0.75)
        ac.ret_oms.std.fill_(3.0)
        for net in (ac.pi, ac.v):
            for m in net:
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
    ac.set_log_std(0.4)
    return env, twin, ac, RolloutCollector(env, ac, T, reset_each_rollout=reset_each)


def _perturb(ac):
    """An optimiser step's worth of change, in place (the packed image must follow)."""
    with torch.no_grad():
        for p_ in list(ac.pi.parameters()) + list(ac.v.parameters()):
            if p_.requires_grad:
                p_.add_(0.02 * torch.randn_like(p_))


def _run(env, twin, ac, col, n_collects, label):
    """n_collects rollouts with what PPO does in between; checks each and the continuation invariants."""
    reports, prev_last = [], None
    for k in range(n_collects):
        snap = snapshot(ac, env)
        reset = col.reset_each_rollout or not col._started
        data = col.collect()
        assert ac._counter - snap['c0'] == (0 if env.dtype == torch.float64 else col.T), label
        assert env._counter - snap['env_counter'] == col.T + (1 if reset else 0), label
        if prev_last is not None and not reset:
            assert torch.equal(col.obs[0], prev_last), (label, 'obs[0] must continue from obs[T]')
        prev_last = col.obs[col.T].clone()
        reports.append(check_rollout(col, data, twin, snap, reset, f'{label} #{k}'))
        col.update_running_statistics(data)
        _perturb(ac)
    return reports


def _print(label, reports):
    for k, r in enumerate(reports):
        print(f'{label} #{k}: fused_used={r["fused_used"]} tc_precision={r["tc_precision"]} policy {r["policy"]:.2e} '
              f'tf32 mu {r["tf32_mu"]:.2e} v-bound residual {r["tf32_v"]:.2e} env {r["env"]:.2e} truncations {r["trunc"]}')


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tensor_core_plan_accepts(env, ac):
    """pdx_collect reads the weight image of the stand-alone tensor-core kernel.  That kernel's shared-memory plan has
    no room for the two split-TF32 images of rows wider than 48 (D = 51, 60): pdx_policy_tc_pack_words refuses them
    with PDX_ERR_INVALID, the ActorCritic takes the CUDA-core kernel and the collector alternates launches."""
    import ctypes as C
    from phoenix_drone_simulation_b200 import lib as _lib
    pi, v = ac._mlp_struct(ac.pi, ac.log_std.shape[0]), ac._mlp_struct(ac.v, 1)
    words = int(_lib.load().pdx_policy_tc_pack_words(env.obs_dim, C.byref(pi), C.byref(v), ac.tc_precision))
    assert words > 0 or words == -1, words                                    # -1: PDX_ERR_INVALID
    return words > 0


def _assert_path(env, ac, accepted, report, label):
    if accepted:
        assert report['fused_used'] and ac.tc_precision in (1, 3), (label, report)
    else:
        assert not report['fused_used'] and ac.tc_precision == 0, (label, report)


# ---------------------------------------------------------------------------------------------
#  continuing episodes and time limits through pdx_collect
# ---------------------------------------------------------------------------------------------
CONTINUE_CASES = [
    ('DroneHoverSimpleEnv-v0', 'tc', 1000, 16, False, dict(max_episode_steps=7)),
    ('DroneHoverBulletEnv-v0', 'tc_tf32', 5000, 24, False, dict(max_episode_steps=10)),
    ('DroneCircleBulletEnv-v0', 'tc', 'two_passes', 8, False, dict(max_episode_steps=5)),
    ('DroneCircleSimpleEnv-v0', 'tc', 33, 16, False, dict(reset_on_nonfinite=True, max_episode_steps=6)),
    ('DroneHoverBulletEnv-v0', 'tc', 2000, 12, True, dict(max_episode_steps=12)),     # truncation at the last step
]


@pytest.mark.parametrize('env_id,kernel,N,T,reset_each,kw', CONTINUE_CASES)
def test_fused_collector_continues_episodes_across_rollouts(env_id, kernel, N, T, reset_each, kw):
    torch.manual_seed(4)
    if N == 'two_passes':
        N = _sms() * 448 + 1000                       # more environments than one pass of 14-warp CTAs holds
    env, twin, ac, col = _make(env_id, kernel, N, T, reset_each, **kw)
    label = f'{env_id} [{kernel}] N={N} T={T}'
    reports = _run(env, twin, ac, col, 3, label)
    _print(label, reports)
    for r in reports:
        assert r['fused_used'] and r['trunc'] > 0, (label, r)


# ---------------------------------------------------------------------------------------------
#  the alternating-launch fallback
# ---------------------------------------------------------------------------------------------
FALLBACK_CASES = [
    ('DroneTakeOffSimpleEnv-v0', 'tc', {}, dict(reset_on_nonfinite=True), 3),
    ('DroneTakeOffBulletEnv-v0', 'tc_tf32', {}, {}, 1),
    ('DroneHoverBulletEnv-v0', 'tc_tf32', {}, dict(control_mode='AttitudeRate'), 1),
    ('DroneCircleSimpleEnv-v0', 'tc', {}, dict(observation_history_size=8), 0),
    ('DroneHoverSimpleEnv-v0', 'tc', dict(pi_hidden=(64, 64)), {}, 3),
    ('DroneHoverSimpleEnv-v0', 'tc', {}, dict(observation_noise=0), 3),
    ('DroneHoverSimpleEnv-v0', 'tc', dict(dtype=torch.float64), {}, 3),
    ('DroneHoverBulletEnv-v0', 'tc', {}, {}, 3),
]


@pytest.mark.parametrize('env_id,kernel,make_kw,env_kw,precision', FALLBACK_CASES)
def test_alternating_collector_matches_reference(env_id, kernel, make_kw, env_kw, precision):
    torch.manual_seed(6)
    N, T = 600, 10
    env, twin, ac, col = _make(env_id, kernel, N, T, False, max_episode_steps=6, **make_kw, **env_kw)
    unforced = not make_kw and not env_kw and env_id == 'DroneHoverBulletEnv-v0'
    if unforced:
        col.use_fused_kernel = False                  # the same configuration as a fused case
    label = f'{env_id} [{kernel}] {make_kw} {env_kw}'
    reports = _run(env, twin, ac, col, 2, label)
    _print(label, reports)
    for r in reports:
        assert not r['fused_used'] and r['trunc'] > 0, (label, r)
    assert ac.tc_precision == precision, (label, ac.tc_precision)
    if unforced:                                      # step 0 agrees with pdx_collect from the same seeds
        torch.manual_seed(6)
        env_f, _, ac_f, col_f = _make(env_id, kernel, N, T, False, max_episode_steps=6)
        env_a, _, ac_a, col_a = _make(env_id, kernel, N, T, False, max_episode_steps=6)
        ac_f.load_state_dict(ac_a.state_dict())
        col_a.use_fused_kernel = False
        col_f.collect(); col_a.collect()
        assert col_f.fused_used and not col_a.fused_used
        assert torch.equal(col_f.obs[0], col_a.obs[0])
        for x, y in ((col_f.act[0], col_a.act[0]), (col_f.val[0], col_a.val[0])):
            assert _rel(x.double().cpu().numpy(), y.double().cpu().numpy()) <= TOL_F32
        assert _rel(col_f.obs[1].double().cpu().numpy(), col_a.obs[1].double().cpu().numpy()) <= TOL_ENV


# ---------------------------------------------------------------------------------------------
#  pdx_collect across the observation widths and networks it accepts
# ---------------------------------------------------------------------------------------------
WIDTHS = [('DroneHoverSimpleEnv-v0', 1), ('DroneHoverSimpleEnv-v0', 3), ('DroneHoverBulletEnv-v0', 3),
          ('DroneCircleSimpleEnv-v0', 1), ('DroneCircleSimpleEnv-v0', 3)]
NETWORKS = [((50, 50), (64, 64)),
            ((63, 64), (64, 64)),       # the constant-1 unit is the last column of its 8-column group
            ((56, 17), (64, 1)),        # pi_h1 % 8 == 0: the constant unit starts a group
            ((8, 4), (3, 64)),
            ((1, 2), (1, 1))]


@pytest.mark.parametrize('kernel', ['tc', 'tc_tf32'])
@pytest.mark.parametrize('pi_hidden,v_hidden', NETWORKS)
@pytest.mark.parametrize('env_id,history', WIDTHS)
def test_fused_collector_shapes(env_id, history, pi_hidden, v_hidden, kernel):
    torch.manual_seed(8)
    N, T = 300, 8
    env, twin, ac, col = _make(env_id, kernel, N, T, False, pi_hidden=pi_hidden, v_hidden=v_hidden,
                               observation_history_size=history, max_episode_steps=5)
    label = f'{env_id} H={history} D={env.obs_dim} pi {pi_hidden} v {v_hidden} [{kernel}]'
    accepted = _tensor_core_plan_accepts(env, ac)
    assert accepted or (kernel == 'tc' and env.obs_dim > 48), label
    reports = _run(env, twin, ac, col, 1, label)
    _print(label, reports)
    _assert_path(env, ac, accepted, reports[0], label)
    assert reports[0]['trunc'] > 0, label


@pytest.mark.parametrize('kernel', ['tc', 'tc_tf32'])
@pytest.mark.parametrize('env_id,history', [('DroneCircleSimpleEnv-v0', 2), ('DroneCircleSimpleEnv-v0', 3),
                                            ('DroneHoverBulletEnv-v0', 3)])
def test_fused_collector_wide_rows_at_full_occupancy(env_id, history, kernel):
    """Shards that ask for 14 warps per CTA with rows whose shared-memory plan admits fewer (D = 40 with split-TF32
    images: 10 warps; D = 60 with single TF32: 11): pdx_collect takes more passes instead of failing the launch."""
    torch.manual_seed(9)
    N, T = _sms() * 448, 4
    env, twin, ac, col = _make(env_id, kernel, N, T, False, observation_history_size=history, max_episode_steps=3)
    label = f'{env_id} H={history} D={env.obs_dim} N={N} [{kernel}]'
    accepted = _tensor_core_plan_accepts(env, ac)
    assert accepted or (kernel == 'tc' and env.obs_dim > 48), label
    reports = _run(env, twin, ac, col, 1, label)
    _print(label, reports)
    _assert_path(env, ac, accepted, reports[0], label)
    assert reports[0]['trunc'] > 0, label


def test_single_tf32_reference_model():
    """Which conversion the tensor core applies to pdx_collect's raw float32 operands (X, layer-1 activations) in
    single-TF32 mode: the actor mean of a DroneHoverBulletEnv-v0 rollout (5,000 environments, 8 steps) against the
    model with truncated and with rounded operands.  The kernel's mean is recovered as act - std * draw.
    Measured on a B200 (1,000 W): truncated 1.0e-4, rounded 4.5e-4 (see COLLECT_TF32_CONVERT)."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic
    torch.manual_seed(10)
    N, T = 5000, 8
    env, _, ac, col = _make('DroneHoverBulletEnv-v0', 'tc_tf32', N, T, True)
    snap = snapshot(ac, env)
    col.collect()
    assert col.fused_used and ac.tc_precision == 1
    draw_ac = ActorCritic(env.obs_dim, seed=ac.seed, policy_kernel='cuda')
    draw_ac.load_state_dict(snap['sd'])
    draw_ac.env_offset = ac.env_offset
    a2 = torch.empty((N, 4), device='cuda'); v2 = torch.empty(N, device='cuda')
    l2 = torch.empty(N, device='cuda'); m2 = torch.empty((N, 4), device='cuda')
    err = {'trunc': [0.0, 0.0], 'rna': [0.0, 0.0]}
    for t in range(T):
        draw_ac._launch_into(col.obs[t].contiguous(), a2, v2, l2, m2, counter=snap['c0'] + 1 + t)
        mu_k = (col.act[t].double() - (a2.double() - m2.double())).cpu().numpy()       # act - std * draw
        rows = col.obs[t].double().cpu().numpy()
        v_k = col.val[t].double().cpu().numpy()
        for mode in err:
            mu, v, terms = tfr.forward(rows, snap['mean'], snap['std'], snap['eps'], snap['pi'], snap['v'], mode)
            err[mode][0] = max(err[mode][0], float(np.abs(mu_k - mu).max()))
            err[mode][1] = max(err[mode][1], float((np.abs(v_k - v) - tfr.tanh_bound(terms)).max()))
    print('single TF32, pdx_collect vs model: ' + ', '.join(f'{m}: mu {e[0]:.2e}, v residual {e[1]:.2e}' for m, e in err.items()))
    other = 'rna' if COLLECT_TF32_CONVERT == 'trunc' else 'trunc'
    assert err[COLLECT_TF32_CONVERT][0] <= TOL_TF32_MU and err[COLLECT_TF32_CONVERT][1] <= TOL_TF32_V
    assert 2 * err[COLLECT_TF32_CONVERT][0] < err[other][0], err          # the pinned model is the one that fits
