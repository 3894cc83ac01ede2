"""GPU tests of the rollout-collector kernels (pdx_gae, pdx_moments) and of the device-side
collector, against oracle/collector_oracle.py and the reference's golden vectors
(tests/golden_collector).  float32 arithmetic: tolerance 2e-4 relative / absolute (the kernel walks
time backwards in float32 like scipy.lfilter does, summation order identical, FMA contraction
allowed)."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import collector_oracle as co
import tf32_reference as tfr

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden_collector')


def _load(name):
    z = np.load(os.path.join(GOLD, name + '.npz'))
    return {k: z[k] for k in z.files}


def _cuda(x):
    return torch.as_tensor(x, device='cuda')


@pytest.mark.parametrize('name', ['gae_scaled', 'gae_plain'])
def test_gae_kernel_matches_reference_golden(name):
    from phoenix_drone_simulation_b200.rollout import compute_gae
    g = _load(name)
    ret_std = float(g['ret_std'][0]) if bool(g['scaled']) else None
    col = lambda k: _cuda(g[k])[:, None].repeat(1, 5).contiguous()
    adv, tv, dr = compute_gae(col('rew'), col('val'), col('done'), col('boot_val'),
                              _cuda(np.full(5, g['last_val'], np.float32)), 0.99, 0.95, ret_std)
    for got, ref in ((adv, g['adv']), (tv, g['target_v']), (dr, g['disc_ret'])):
        for c in range(5):
            np.testing.assert_allclose(got[:, c].cpu().numpy(), ref, rtol=2e-4, atol=2e-4)


def test_gae_kernel_matches_oracle_on_random_rollout():
    from phoenix_drone_simulation_b200.rollout import compute_gae
    rng = np.random.default_rng(7)
    T, N = 70, 300
    rew = rng.normal(-1, 2, (T, N)).astype(np.float32)
    val = rng.normal(-5, 3, (T, N)).astype(np.float32)
    u = rng.random((T, N))
    done = np.where(u < 0.05, 1, np.where(u < 0.08, 2, 0)).astype(np.uint8)
    boot = (rng.normal(-5, 3, (T, N)) * (done == 2)).astype(np.float32)
    last = rng.normal(-5, 3, N).astype(np.float32)
    for ret_std in (None, 17.5):
        adv, tv, dr = compute_gae(_cuda(rew), _cuda(val), _cuda(done), _cuda(boot), _cuda(last), 0.99, 0.95, ret_std)
        a0, t0, d0 = co.rollout_gae(rew, val, done, boot, last, 0.99, 0.95, ret_std)
        np.testing.assert_allclose(adv.cpu().numpy(), a0, rtol=2e-4, atol=2e-4)
        np.testing.assert_allclose(tv.cpu().numpy(), t0, rtol=2e-4, atol=2e-4)
        np.testing.assert_allclose(dr.cpu().numpy(), d0, rtol=2e-4, atol=2e-4)


def test_moments_kernel():
    from phoenix_drone_simulation_b200.rollout import column_moments
    g = torch.Generator(device='cuda').manual_seed(0)
    for rows, dim in ((1, 1), (1000, 34), (4097, 160), (65536, 48), (333, 1)):
        x = torch.randn((rows, dim), device='cuda', generator=g) * 3 + 1
        sh = torch.randn(dim, device='cuda', generator=g, dtype=torch.float64)
        s1, s2 = column_moments(x, sh)
        xd = x.double()
        torch.testing.assert_close(s1, xd.sum(0), rtol=1e-10, atol=1e-8)
        torch.testing.assert_close(s2, ((xd - sh) ** 2).sum(0), rtol=1e-10, atol=1e-8)
        s1b, s2b = column_moments(x, None)
        torch.testing.assert_close(s2b, (xd ** 2).sum(0), rtol=1e-10, atol=1e-8)


@pytest.mark.parametrize('name', ['oms_obs34', 'oms_ret1'])
def test_online_mean_std_on_device_matches_reference(name):
    from phoenix_drone_simulation_b200.rollout import OnlineMeanStd
    g = _load(name)
    dim = g['x'].shape[2]
    oms = OnlineMeanStd(dim, 'cuda')
    for b in range(g['x'].shape[0]):
        oms.update(_cuda(g['x'][b]))
        np.testing.assert_allclose(oms.mean.cpu().numpy(), g['mean'][b], rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(oms.std.cpu().numpy(), g['std'][b], rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(oms.count.cpu().numpy(), g['count'][b])
    np.testing.assert_allclose(oms(_cuda(g['probe'])).cpu().numpy(), g['forward'], rtol=1e-4, atol=1e-5)


# k_policy_tc with single-TF32 operands (it rounds X and the hidden activations to nearest itself) against the
# float64 model of those operands (tests/tf32_reference.py), |got - model| / (1 + |model|) for the mean; the value
# adds the tanh.approx bound of its layer-2 activations per row.  Measured on a B200 (1,000 W): mean at most 1.3e-4
# (2.4e-7 on the check-sum networks), value at most 3.4e-4 inside the tanh bound.  Tolerances: about 4x.
TF32_RNA_MU = 6e-4
TF32_RNA_V = 2e-4


def _net_layers(net):
    return [(m.weight.detach().cpu().numpy(), m.bias.detach().cpu().numpy()) for m in net if isinstance(m, torch.nn.Linear)]


def _check_single_tf32(ac, obs, mu, val, label):
    oms = ac.obs_oms
    mean, std = (oms.mean.cpu().numpy(), oms.std.cpu().numpy()) if oms is not None else (None, None)
    mu_m, v_m, terms = tfr.forward(obs.cpu().numpy(), mean, std, oms.eps if oms is not None else 0.0,
                                   _net_layers(ac.pi), _net_layers(ac.v), 'rna')
    n_out = mu_m.shape[1]
    e_mu = float((np.abs(mu[:, :n_out].double().cpu().numpy() - mu_m) / (1 + np.abs(mu_m))).max())
    e_v = float((np.abs(val.double().cpu().numpy() - v_m) - tfr.tanh_bound(terms)).max())
    print(f'single TF32 {label}: mean vs model {e_mu:.2e}, value vs model beyond the tanh bound {e_v:.2e}')
    assert e_mu <= TF32_RNA_MU and e_v <= TF32_RNA_V, (label, e_mu, e_v)
    return mu_m


@pytest.mark.parametrize('kernel', ['cuda', 'tc', 'tc_tf32'])
def test_fused_policy_step_matches_torch_modules(kernel):
    """pdx_policy_step / pdx_policy_step_tc (standardise + actor MLP + critic MLP + sample + log-prob in
    one kernel) against the torch modules that own the weights.  'cuda' = CUDA-core float32 kernel and
    'tc' = tcgen05 tensor-core kernel with split-TF32 operands: tolerance 2e-5 abs on mean / value;
    'tc_tf32' = single TF32 rounding of the operands: against the model of those operands (_check_single_tf32)."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic
    torch.manual_seed(1)
    tol = dict(rtol=1e-4, atol=2e-5)                    # (single TF32 goes through _check_single_tf32)
    # (160, ...) is outside the tensor-core shared-memory plan: ActorCritic falls back to the CUDA-core kernel
    for obs_dim, pi_h, v_h, n in ((34, (50, 50), (64, 64), 5000), (160, (64, 64), (64, 32), 777), (17, (8, 50), (3, 64), 256),
                                  (40, (64, 64), (64, 64), 128 * 300 + 1), (48, (50, 50), (64, 64), 127)):
        ac = ActorCritic(obs_dim, pi_hidden=pi_h, v_hidden=v_h, device='cuda', seed=3, policy_kernel=kernel)
        ac.obs_oms.mean.copy_(torch.randn(obs_dim, device='cuda') * 0.3)
        ac.obs_oms.std.copy_(torch.rand(obs_dim, device='cuda') + 0.5)
        ac.set_log_std(0.7)
        obs = torch.randn((n, obs_dim), device='cuda') * 2
        act = torch.empty((n, 4), device='cuda'); val = torch.empty(n, device='cuda'); logp = torch.empty(n, device='cuda')
        mu = torch.empty((n, 4), device='cuda')
        ac.step_into(obs, act, val, logp, mu)
        assert ac.tc_precision == ({'cuda': 0, 'tc': 3, 'tc_tf32': 1}[kernel] if obs_dim <= 64 else 0)
        o = ac.obs_oms(obs)
        if ac.tc_precision == 1:
            _check_single_tf32(ac, obs, mu, val, f'D={obs_dim} pi {pi_h} v {v_h}')
        else:
            torch.testing.assert_close(mu, ac.pi(o), **tol)
            torch.testing.assert_close(val, ac.v(o).squeeze(-1), **tol)
        std = torch.exp(ac.log_std)
        ref_logp = torch.distributions.Normal(mu, std).log_prob(act).sum(-1)
        torch.testing.assert_close(logp, ref_logp, rtol=1e-4, atol=1e-4)
        z = ((act - mu) / std).flatten()
        if n >= 5000:
            assert abs(float(z.mean())) < 0.03 and abs(float(z.std()) - 1) < 0.03
        act2 = torch.empty_like(act)
        ac.step_into(obs, act2, val, logp)                      # next counter -> new draws
        assert not torch.equal(act, act2)


def test_tensor_core_policy_draws_and_updates_follow_the_cuda_core_kernel():
    """Both policy kernels use the same Philox counters and the same Box-Muller: for equal (seed,
    counter) the standardised draws (a - mu) / std agree to float32 rounding.  An in-place weight update
    must reach the packed tensor-core image (torch bumps the parameter version)."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic
    torch.manual_seed(5)
    n, d = 4099, 34
    acs = {k: ActorCritic(d, device='cuda', seed=9, policy_kernel=k) for k in ('cuda', 'tc')}
    acs['tc'].load_state_dict(acs['cuda'].state_dict())
    obs = torch.randn((n, d), device='cuda')
    out = {}
    for k, ac in acs.items():
        act = torch.empty((n, 4), device='cuda'); val = torch.empty(n, device='cuda'); logp = torch.empty(n, device='cuda')
        mu = torch.empty((n, 4), device='cuda')
        ac.step_into(obs, act, val, logp, mu)
        out[k] = (act, val, logp, mu)
    torch.testing.assert_close(out['tc'][3], out['cuda'][3], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(out['tc'][1], out['cuda'][1], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(out['tc'][0] - out['tc'][3], out['cuda'][0] - out['cuda'][3], rtol=0, atol=1e-5)
    torch.testing.assert_close(out['tc'][2], out['cuda'][2], rtol=0, atol=1e-5)
    ac = acs['tc']
    with torch.no_grad():
        for p_ in ac.pi.parameters():
            p_.add_(0.05 * torch.randn_like(p_))
    act = torch.empty((n, 4), device='cuda'); val = torch.empty(n, device='cuda'); logp = torch.empty(n, device='cuda')
    mu = torch.empty((n, 4), device='cuda')
    ac.step_into(obs, act, val, logp, mu)
    torch.testing.assert_close(mu, ac.pi(ac.obs_oms(obs)), rtol=1e-4, atol=2e-5)
    assert not torch.allclose(mu, out['tc'][3], atol=1e-3)
    # an observation buffer that is only 4-byte aligned: no TMA bulk copies, the epilogue warps stage the tiles
    flat = torch.empty(n * d + 1, device='cuda')
    obs_u = flat[1:].view(n, d)
    obs_u.copy_(obs)
    assert obs_u.data_ptr() % 16 == 4 and obs_u.is_contiguous()
    mu_u = torch.empty_like(mu)
    ac.step_into(obs_u, act, val, logp, mu_u)
    torch.testing.assert_close(mu_u, mu, rtol=0, atol=0)


@pytest.mark.parametrize('kernel', ['cuda', 'tc'])
def test_policy_kernels_match_the_numpy_oracle(kernel):
    """Both policy kernels against oracle.actor_critic_step (float64 numpy restatement of ActorCritic.step,
    pinned to the reference loader's golden): mean, value, and -- replaying the draw the kernel made --
    action and log-probability.  float32 kernels: 2e-5 abs."""
    from phoenix_drone_simulation_b200.rollout import ActorCritic
    torch.manual_seed(11)
    n, d = 3000, 34
    ac = ActorCritic(d, device='cuda', seed=2, policy_kernel=kernel)
    ac.obs_oms.mean.copy_(torch.randn(d, device='cuda') * 0.2)
    ac.obs_oms.std.copy_(torch.rand(d, device='cuda') + 0.5)
    ac.set_log_std(0.6)
    obs = torch.randn((n, d), device='cuda') * 1.5
    act = torch.empty((n, 4), device='cuda'); val = torch.empty(n, device='cuda'); logp = torch.empty(n, device='cuda')
    mu = torch.empty((n, 4), device='cuda')
    ac.step_into(obs, act, val, logp, mu)
    layers = lambda net: [(m.weight.detach().cpu().numpy(), m.bias.detach().cpu().numpy()) for m in net if isinstance(m, torch.nn.Linear)]
    log_std = ac.log_std.detach().cpu().numpy()
    draw = ((act - mu) / torch.exp(ac.log_std)).cpu().numpy().astype(np.float64)      # the standardised draw the kernel used
    a_o, v_o, lp_o, mu_o = co.actor_critic_step(obs.cpu().numpy(), ac.obs_oms.mean.cpu().numpy(), ac.obs_oms.std.cpu().numpy(),
                                                layers(ac.pi), layers(ac.v), log_std, draw, norm_eps=ac.obs_oms.eps)
    np.testing.assert_allclose(mu.cpu().numpy(), mu_o, rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(val.cpu().numpy(), v_o, rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(act.cpu().numpy(), a_o, rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(logp.cpu().numpy(), lp_o, rtol=1e-4, atol=1e-4)
    assert abs(draw.mean()) < 0.05 and abs(draw.std() - 1) < 0.05


def test_collector_end_to_end_config5():
    """BASELINE config 5: DroneHoverBulletEnv-v0 driving a PPO rollout (reference networks), all on
    device.  Checks the stored fields against an independent recomputation."""
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
    torch.manual_seed(0)
    N, T = 2048, 48
    env = VecEnv('DroneHoverBulletEnv-v0', N, seed=5, keep_final_obs=True)
    ac = ActorCritic(env.obs_dim, device='cuda')
    col = RolloutCollector(env, ac, T)
    data = col.collect()
    assert data['obs'].shape == (T, N, env.obs_dim) and data['act'].shape == (T, N, 4)
    for k in ('obs', 'act', 'adv', 'target_v', 'log_p', 'discounted_ret'):
        assert torch.isfinite(data[k]).all(), k
    # values / log-probs are those of the stored (obs, act)
    v = ac.value(data['obs'][7])
    torch.testing.assert_close(v, data['val'][7], rtol=1e-5, atol=1e-5)
    mu = ac.pi(ac.obs_oms(data['obs'][7].float()))
    logp = torch.distributions.Normal(mu, torch.exp(ac.log_std)).log_prob(data['act'][7]).sum(-1)
    torch.testing.assert_close(logp, data['log_p'][7], rtol=1e-4, atol=1e-4)
    # GAE of a few columns against the oracle
    done = data['done'].cpu().numpy()
    last_val = ac.value(col.obs[T]).cpu().numpy()
    cols = [0, 5, 777, N - 1]
    a0, t0, d0 = co.rollout_gae(data['rew'].float().cpu().numpy()[:, cols], data['val'].cpu().numpy()[:, cols],
                                done[:, cols], col.boot.cpu().numpy()[:, cols], last_val[cols], 0.99, 0.95,
                                float(ac.ret_oms.std))
    np.testing.assert_allclose(data['adv'].cpu().numpy()[:, cols], a0, rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(data['discounted_ret'].cpu().numpy()[:, cols], d0, rtol=2e-4, atol=2e-4)
    # episode statistics = what the flags say
    es = data['episode_stats']
    assert es.n == int((done != 0).sum())
    if es.n:
        assert es.ret_min <= es.ret_mean <= es.ret_max and 1 <= es.len_min <= es.len_max <= T
    # running statistics update (two moment passes on device)
    col.update_running_statistics(data)
    o = data['obs'].reshape(-1, env.obs_dim).float()
    torch.testing.assert_close(ac.obs_oms.mean, o.mean(0), rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(ac.obs_oms.std, o.std(0, unbiased=False), rtol=1e-3, atol=1e-4)
    data2 = col.collect()           # second rollout uses the updated normaliser
    assert torch.isfinite(data2['adv']).all()


def test_ppo_learns_to_hover():
    """End-to-end sanity of engine + collector + GAE + update: PPO (reference hyper-parameters,
    algs/iwpg/iwpg.py:26-60) on DroneHoverSimpleEnv-v0.  Within twelve epochs of 4,096 x 64 steps the
    number of episodes that END inside a 64-step rollout must fall below a quarter of the initial
    count (observed: 28,955 -> ~700; after 30 epochs ~20)."""
    from phoenix_drone_simulation_b200.ppo import PPO
    alg = PPO('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=12, seed=0)
    alg.learn()
    first, last = alg.history[0], alg.history[-1]
    assert all(math.isfinite(r['loss_v']) and math.isfinite(r['loss_pi']) for r in alg.history)
    assert last['episodes'] < 0.25 * first['episodes'], (first, last)
    assert last['EpLen'] > 2 * first['EpLen']


def test_policy_json_on_device_and_batched_evaluator():
    """The JSON golden (reference loader output) through the fused policy kernel, and the batched
    EnvironmentEvaluator (utils/evaluation.py:52-107): deterministic, repeatable, sane ranges."""
    from phoenix_drone_simulation_b200.policy_io import load_policy_json, evaluate
    g = _load('policy_json')
    ac = load_policy_json(os.path.join(GOLD, 'policy_json.json'), device='cuda')
    n = g['obs'].shape[0]
    act = torch.empty((n, 4), device='cuda'); val = torch.empty(n, device='cuda'); logp = torch.empty(n, device='cuda')
    mu = torch.empty((n, 4), device='cuda')
    ac.step_into(_cuda(g['obs']), act, val, logp, mu)
    np.testing.assert_allclose(mu.cpu().numpy(), g['mu'], rtol=1e-4, atol=2e-5)
    r1, l1, c1 = evaluate('DroneHoverSimpleEnv-v0', ac, num_evaluations=128, seed=3)
    r2, l2, c2 = evaluate('DroneHoverSimpleEnv-v0', ac, num_evaluations=128, seed=3)
    assert r1.shape == (128,) and np.isfinite(r1).all() and (l1 >= 1).all() and (l1 <= 500).all()
    np.testing.assert_array_equal(r1, r2)
    np.testing.assert_array_equal(l1, l2)
    assert (r1 < 0).all() and (c1 >= 0).all()


def test_simopt_objective_recovers_motor_parameters():
    """simopt/pybullet.py:72-225 on the batched engine.  "Flight logs" come from the engine itself run
    with known motor parameters (thrust-to-weight 1.95, motor time constant 60 ms); the objective,
    evaluated for a grid of candidates in one fused launch, must be ~0 at the truth and minimal there."""
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.simopt import TrajectoryObjective, euler_from_quat
    true_t2w, true_tau, M, T, P = 1.95, 0.060, 24, 35, 5
    kw = dict(domain_randomization=-1, observation_noise=-1, motor_thrust_noise=0.0, auto_reset=False,
              enable_reset_distribution=False)
    env = VecEnv('DroneHoverBulletEnv-v0', M, dtype=torch.float64, seed=1, **kw)
    env.reset()
    ts = env.pdx.time_step
    env.set_state('motor_b', torch.full((M, 4), ts / true_tau, dtype=torch.float64))
    env.set_state('motor_k', torch.full((M, 4), 0.028 * 9.81 * true_t2w / 4, dtype=torch.float64))
    g = torch.Generator(device='cuda').manual_seed(5)
    acts = (0.11 + 0.15 * torch.randn((P + T, M, 4), device='cuda', generator=g)).clamp(-1, 1).float()
    logs = []
    for t in range(P + T):
        o, _, _, _, _ = env.step(acts[t])
        e0 = env.core_dim + 4                                # newest history entry (H = 2) starts here
        c = o[:, e0:e0 + 13].double()                        # noise off: xyz, quat, vel, body rates
        logs.append(torch.cat([c[:, 0:3], c[:, 7:10], euler_from_quat(c[:, 3:7]), c[:, 10:13]], dim=1))
    logs = torch.stack(logs, dim=1)                          # [M, P+T, 12], state AFTER step t
    # mini-trajectory: observation 0 = state after step P-1; action i drives observation i -> i+1
    # (the latency ring and the motor lag make the real system depend on earlier inputs, which is
    # exactly why the reference replays pre-steps; a cleared ring leaves a small irreducible loss)
    observations = logs[:, P - 1:P - 1 + T]
    actions = acts[P:P + T].transpose(0, 1)
    pre_inputs = acts[:P].transpose(0, 1)
    obj = TrajectoryObjective(observations.cpu().numpy(), actions.cpu().numpy(), pre_inputs.cpu().numpy(),
                              motor_thrust_noise=0.0, enable_reset_distribution=False)
    t2ws = [1.6, 1.8, 1.95, 2.1, 2.3]
    taus = [0.03, 0.06, 0.12]
    cands = [(a, b) for a in t2ws for b in taus]
    loss = obj.evaluate(cands).cpu().numpy()
    best = cands[int(loss.argmin())]
    assert best[0] == true_t2w, (best, loss)
    assert np.isfinite(loss).all() and loss.min() < 0.5 * np.median(loss)


def test_stats_combine_kernel():
    """pdx_stats_combine (utils/mpi_tools.py:217-240 across ranks): sums of words 0..3, minima of 4 and 6,
    maxima of 5 and 7 over the gathered per-rank vectors."""
    import ctypes as C
    from phoenix_drone_simulation_b200 import lib as _lib
    rng = np.random.default_rng(3)
    for world in (1, 2, 8):
        g = rng.normal(0, 50, (world, 8))
        g[:, 0] = rng.integers(0, 100, world)
        gathered = torch.as_tensor(g, device='cuda').contiguous()
        out = torch.zeros(8, dtype=torch.float64, device='cuda')
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.load().pdx_stats_combine(world, C.c_void_p(gathered.data_ptr()), C.c_void_p(out.data_ptr()), st))
        ref = np.concatenate([g[:, :4].sum(0), [g[:, 4].min(), g[:, 5].max(), g[:, 6].min(), g[:, 7].max()]])
        np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-14, atol=1e-12)


def _nccl_worker(rank, world, port, batches, ep, out_q):
    import torch.distributed as dist
    from phoenix_drone_simulation_b200.rollout import (OnlineMeanStd, allreduce_episode_stats, gather_episode_stats_async,
                                                       EpisodeStats)
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', init_method=f'tcp://127.0.0.1:{port}', rank=rank, world_size=world, device_id=dev)
    dim = batches[0][0].shape[1]
    oms = OnlineMeanStd(dim, dev, dist=dist)                      # CUDA moments kernel + NCCL all-reduces
    for b in batches:
        oms.update(torch.as_tensor(b[rank], device=dev))
    x = np.asarray(ep[rank], np.float64)
    vec = [len(x), x.sum(), (x ** 2).sum(), 3.0 * len(x), x.min(), x.max(), 7.0 + rank, 100.0 + rank]
    stats = torch.tensor(vec, dtype=torch.float64, device=dev)
    allreduce_episode_stats(stats, dist)                          # all-gather + pdx_stats_combine
    later = gather_episode_stats_async(torch.tensor(vec, dtype=torch.float64, device=dev), dist)
    torch.zeros(1 << 20, device=dev).add_(1)                      # unrelated work between start and finish
    stats2 = later()
    es = EpisodeStats(stats)
    out_q.put((rank, oms.mean.cpu().numpy(), oms.std.cpu().numpy(), float(oms.count), es.as_dict(), es.len_min, es.len_max,
               stats2.cpu().numpy(), stats.cpu().numpy()))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_nccl_world2_running_stats_and_episode_stats():
    """The NCCL branch of OnlineMeanStd._avg and pdx_stats_combine behind one NCCL all-gather, world size 2,
    against the oracle -- the same expectations as the gloo test of tests/test_collector_oracle.py."""
    import socket
    import torch.multiprocessing as mp
    rng = np.random.default_rng(0)
    world, dim = 2, 6
    batches = [[rng.normal(b, 1 + b, (32, dim)).astype(np.float32) for _ in range(world)] for b in range(3)]
    ep = [rng.normal(-50, 20, 11).astype(np.float32), rng.normal(-80, 5, 5).astype(np.float32)]
    s = socket.socket(); s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, batches, ep, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(world)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    o = co.OnlineMeanStdOracle(dim)
    for b in batches:
        o.update(b)
    mean, std, mn, mx = co.statistics_scalar(ep)
    for _, m, s_, c, d, lmin, lmax, async_stats, sync_stats in res:
        np.testing.assert_allclose(m, o.mean, rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(s_, o.std, rtol=2e-5, atol=1e-6)
        assert c == float(o.count[0]) == 3 * 32 * world
        assert d['Episodes'] == 16
        assert abs(d['EpRet/Mean'] - mean) < 1e-3 and abs(d['EpRet/Std'] - std) < 1e-2
        assert abs(d['EpRet/Min'] - mn) < 1e-4 and abs(d['EpRet/Max'] - mx) < 1e-4
        assert (lmin, lmax) == (7.0, 101.0)
        np.testing.assert_array_equal(async_stats, sync_stats)      # asynchronous form == synchronous form
    np.testing.assert_array_equal(res[0][1], res[1][1])
    np.testing.assert_array_equal(res[0][2], res[1][2])


KAT_DIR = os.path.join(GOLD, 'kat_models')


@pytest.mark.parametrize('kernel,tol', [('cuda', 1e-5), ('tc', 1e-5), ('tc_tf32', 5e-3)])
def test_policy_kernels_reproduce_reference_check_sums(kernel, tol):
    """Known-answer test held by the reference itself: for each exported policy, sum(net(ones)) must
    equal the file's check_sum (utils/export.py:47-53, utils/utils.py:324-330).  All three policy kernels
    (CUDA-core float32, tcgen05 split-TF32, tcgen05 single TF32) on six reference-exported networks
    (D = 40, 50-50 relu).  Tolerance: float32 kernels 1e-5 abs + 1e-5 rel (the reference computed the sum
    in float32); single TF32 5e-3 against the check_sum (its operand rounding) and TF32_RNA_MU against the model
    of its operands."""
    from phoenix_drone_simulation_b200.policy_io import load_policy_json, verify_check_sum
    files = sorted(f for f in os.listdir(KAT_DIR) if f.endswith('.json'))
    assert len(files) == 6
    for f in files:
        got, exp = verify_check_sum(os.path.join(KAT_DIR, f), device='cuda', policy_kernel=kernel, rtol=tol, atol=tol)
        print(f'{f} [{kernel}]: kernel {got:.6f} vs check_sum {exp:.6f}')
        if kernel == 'tc_tf32':                   # the same network(ones) against the model of its TF32 operands
            ac = load_policy_json(os.path.join(KAT_DIR, f), device='cuda', standardize=False, policy_kernel=kernel)
            ones = torch.ones((128, ac.pi.net[0].in_features), device='cuda')
            act = torch.empty((128, 4), device='cuda'); val = torch.empty(128, device='cuda')
            logp = torch.empty(128, device='cuda'); mu = torch.empty((128, 4), device='cuda')
            ac.step_into(ones, act, val, logp, mu)
            mu_m = _check_single_tf32(ac, ones, mu, val, f)
            assert abs(got - float(mu_m[0].sum())) <= TF32_RNA_MU * (1 + abs(got)), (f, got, float(mu_m[0].sum()))


@pytest.mark.parametrize('env_id,kernel,N,T', [('DroneHoverBulletEnv-v0', 'tc', 5000, 24), ('DroneHoverBulletEnv-v0', 'tc_tf32', 5000, 24),
                                                ('DroneCircleSimpleEnv-v0', 'tc', 5000, 24), ('DroneHoverSimpleEnv-v0', 'tc_tf32', 5000, 24),
                                                # edge shapes: one environment; two ragged warps whose rows break the 16-byte
                                                # rule of the bulk copy; a partial tile; a one-step rollout; several passes
                                                ('DroneHoverSimpleEnv-v0', 'tc', 1, 40), ('DroneHoverBulletEnv-v0', 'tc', 33, 30),
                                                ('DroneCircleBulletEnv-v0', 'tc_tf32', 130, 1), ('DroneHoverSimpleEnv-v0', 'tc', 140000, 3)])
def test_fused_collector_kernel_is_policy_kernel_plus_env_kernel(env_id, kernel, N, T):
    """pdx_collect (policy networks on the tensor cores + env.step, whole rollout in one launch, state in
    registers) against its two halves run separately:
      * every stored (value, action, log-prob) equals what the stand-alone policy kernel gives on the stored
        observation with the same Philox counter (float32-level kernels 2e-5; single TF32: 1e-2);
      * replaying the stored actions through the single-step env kernel from the same initial state gives the
        stored observations / rewards / flags (same step body, other instantiation: 4e-6 x (1 + |value|), flags
        equal), i.e. IWPGAlgorithm.roll_out's loop (iwpg.py:350-385) was executed in order;
      * last_val = V(obs[T]), episode statistics equal those of the replay.
    5,000 environments: a ragged last tile; T = 24; plus the edge shapes of the parameter list."""
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector
    tol = 2e-5 if kernel == 'tc' else 1e-2
    torch.manual_seed(4)
    env = VecEnv(env_id, N, seed=21, keep_final_obs=True, env_offset=640)
    twin = VecEnv(env_id, N, seed=21, keep_final_obs=True, env_offset=640)
    ac = ActorCritic(env.obs_dim, policy_kernel=kernel, seed=5)
    with torch.no_grad():
        ac.obs_oms.mean.copy_(torch.randn(env.obs_dim, device='cuda') * 0.1)
        ac.obs_oms.std.copy_(torch.rand(env.obs_dim, device='cuda') * 0.5 + 0.75)
        for net in (ac.pi, ac.v):
            for m in net:
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)
    ac.set_log_std(0.4)
    col = RolloutCollector(env, ac, T)
    c0 = ac._counter
    data = col.collect()
    assert col.fused_used, 'pdx_collect was not used'
    assert torch.isfinite(col.obs).all() and torch.isfinite(col.val).all() and torch.isfinite(col.logp).all()
    # ---- policy half
    act2 = torch.empty((N, 4), device='cuda'); val2 = torch.empty(N, device='cuda'); lp2 = torch.empty(N, device='cuda')
    worst_p = 0.0
    for t in range(T):
        ac._launch_into(col.obs[t].contiguous(), act2, val2, lp2, None, counter=c0 + 1 + t)
        worst_p = max(worst_p, float((act2 - col.act[t]).abs().max()), float((val2 - col.val[t]).abs().max()))
        torch.testing.assert_close(lp2, col.logp[t], rtol=1e-5, atol=1e-5)
    assert worst_p <= tol, worst_p
    torch.testing.assert_close(ac.value(col.obs[T].contiguous()), col.last_val, rtol=tol, atol=tol)
    # ---- env half
    assert torch.equal(twin.reset(), col.obs[0])
    worst_e, n_fin = 0.0, 0
    rel = lambda x, y: float(((x - y).abs() / (1.0 + y.abs())).max())
    for t in range(T):
        o, r, te, tr, info = twin.step(col.act[t].contiguous())
        assert torch.equal(te, col.term[t].bool()) and torch.equal(tr, col.trunc[t].bool()), t
        worst_e = max(worst_e, rel(col.obs[t + 1], o), rel(col.rew[t], r))
        assert torch.equal(info['cost'], col.cost[t])
        n_fin += int((te | tr).sum())
    assert worst_e <= 4e-6, worst_e
    assert (n_fin > 0 or N * T < 2000) and data['episode_stats'].n == n_fin == int(twin.episode_stats()[0])
    # the state written back at the end of the pass (the reset-package pool may differ: the fused kernel
    # regenerates packages per 128-environment tile, the step kernel per block)
    for name in ('xyz', 'vel', 'ou', 'last_action', 'ep_length', 'gyro_bias', 'gyro_lpf', 'dt', 'mass'):
        torch.testing.assert_close(env.get_state(name), twin.get_state(name), rtol=1e-5, atol=1e-5)
    assert torch.equal(env.episode_counters()[0], twin.episode_counters()[0])                  # auto-resets consumed
    # ---- the running-statistics sums accumulated in-kernel == a pass over the observations the policy saw
    mom, shift = data['obs_moments']
    x = col.obs[:T].reshape(T * N, -1).double() - shift.double()
    torch.testing.assert_close(mom[:env.obs_dim], x.sum(0), rtol=1e-6, atol=1e-3)
    torch.testing.assert_close(mom[env.obs_dim:], (x * x).sum(0), rtol=1e-6, atol=1e-3)
    ref = ActorCritic(env.obs_dim, seed=5)
    ref.obs_oms.load_state_dict(ac.obs_oms.state_dict())
    col.update_running_statistics(data)
    ref.obs_oms.update(col.obs[:T])
    torch.testing.assert_close(ac.obs_oms.mean, ref.obs_oms.mean, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(ac.obs_oms.std, ref.obs_oms.std, rtol=1e-5, atol=1e-6)
    print(f'{env_id} [{kernel}]: fused vs policy kernel {worst_p:.2e}, fused vs env kernel {worst_e:.2e}, {n_fin} episodes')


def test_simopt_objective_matches_reference_losses():
    """TrajectoryObjective (K candidates x M mini-trajectories in one reset, five single-step launches and ONE fused
    launch) against the losses the UNMODIFIED reference's evaluate_once gave for every (candidate, mini-trajectory)
    pair (simopt/pybullet.py:130-225; tests/golden_collector/simopt_hover.npz).  float64 engine; tolerance 1e-6 on
    losses of 0.1 ... 25 (observed 5e-8): the engine takes float32 actions (the policy's dtype) where the
    reference's objective feeds the logged float64 ones."""
    from phoenix_drone_simulation_b200.simopt import TrajectoryObjective
    g = _load('simopt_hover')
    obj = TrajectoryObjective(g['observations'], g['actions'], g['pre_inputs'], motor_thrust_noise=0.0)
    L = obj.evaluate(g['candidates'][:, :2], per_trajectory=True).cpu().numpy()
    err = np.abs(L - g['losses']).max()
    print(f'simopt: engine vs reference evaluate_once, max abs err {err:.2e} over {L.size} (candidate, trajectory) pairs')
    assert err <= 1e-6
    np.testing.assert_allclose(obj.evaluate(g['candidates'][:, :2]).cpu().numpy(), g['losses'].mean(1), rtol=0, atol=1e-6)


def test_simopt_objective_fits_latency_like_the_reference():
    """Latency as the third fitted parameter (simopt/pybullet.py:248 -> agents.py:388-404): rings of 0, 0, 1, 2, 3, 4, 7
    and 10 sub-steps against the losses of the UNMODIFIED reference (tests/golden_collector/simopt_hover_latency.npz).
    The engine's ring holds one or two sub-steps; longer rings are that ring behind a per-environment delayed action
    sequence (simopt.py).  Tolerance 1e-6 as above (float32 actions)."""
    from phoenix_drone_simulation_b200.simopt import TrajectoryObjective
    g = _load('simopt_hover_latency')
    obj = TrajectoryObjective(g['observations'], g['actions'], g['pre_inputs'], motor_thrust_noise=0.0)
    L = obj.evaluate(g['candidates'], per_trajectory=True).cpu().numpy()
    err = np.abs(L - g['losses']).max(1)
    print('simopt latency candidates: ring lengths', [int(x) for x in g['ring_lengths']], 'max abs err per candidate', ' '.join(f'{e:.1e}' for e in err))
    assert err.max() <= 1e-6
    np.testing.assert_allclose(obj.evaluate(g['candidates']).cpu().numpy(), g['losses'].mean(1), rtol=0, atol=1e-6)
    # latency matters: the candidates that differ only in their ring length have different losses
    assert abs(g['losses'][2].mean() - g['losses'][3].mean()) > 1e-3


def test_engine_reproduces_reference_roll_out_golden():
    """The golden rollout recorded from the UNMODIFIED reference's IWPGAlgorithm.roll_out (iwpg.py:350-385;
    oracle/gen_golden_rollout.py) through the engine's pieces:
      * float64 tape-mode env kernels on the recorded draws and the recorded actions give the observations and
        rewards the reference's Buffer stored, incl. the first observation after every in-rollout reset (1e-6: the
        Buffer holds float32);
      * the policy kernels (CUDA-core float32 and tcgen05 split-TF32) on the stored observations give the stored
        values (2e-5) and the Gaussian means behind the stored actions;
      * pdx_gae on the stored rewards / values with roll_out's episode boundaries gives the stored advantages,
        value targets and discounted returns (2e-4), reward scaling on."""
    from phoenix_drone_simulation_b200 import VecEnv
    from phoenix_drone_simulation_b200.rollout import ActorCritic, compute_gae
    g = _load('rollout_hover_simple')
    T, env_id = int(g['T']), str(g['env_id'])
    dev = torch.device('cuda')
    # ---- env
    env = VecEnv(env_id, 2, dtype=torch.float64, rng='tape', keep_final_obs=True)
    S, R = env.tape_slots['step'], env.tape_slots['reset']
    col = lambda v, slots: torch.as_tensor(np.asarray(v[:slots], dtype=np.float64), device=dev)[:, None].repeat(1, 2).contiguous()
    env.construct_from_tape(col(g['init_tape'], env.tape_slots['init']))
    env.set_tapes(reset=col(g['reset_tape'][0], R))
    o = env.reset()
    np.testing.assert_allclose(o[0].cpu().numpy(), g['obs'][0], rtol=0, atol=1e-6)
    reset_of_step = {int(t): e for e, t in enumerate(g['reset_after'])}
    done = np.zeros(T, np.uint8)
    for t in range(T):
        e = reset_of_step.get(t)
        env.set_tapes(step=col(g['step_tape'][t], S), reset=col(g['reset_tape'][e] if e is not None else np.zeros(R), R))
        o, r, term, trunc, _ = env.step(torch.as_tensor(g['act'][t], device=dev).expand(2, 4).contiguous())
        assert abs(float(r[0]) - float(g['rew'][t])) <= 1e-5 * max(1.0, abs(float(g['rew'][t])))
        ended = bool(term[0] | trunc[0])
        assert ended == (e is not None and t < T - 1) or t == T - 1
        done[t] = 1 if bool(term[0]) else 0
        if t + 1 < T:
            np.testing.assert_allclose(o[0].cpu().numpy(), g['obs'][t + 1], rtol=0, atol=1e-6)
    next_obs = o[0].float()[None].contiguous()               # the observation the epoch cut is bootstrapped from
    # ---- policy
    for kernel, tol in (('cuda', 2e-5), ('tc', 2e-5)):
        ac = ActorCritic(env.obs_dim, policy_kernel=kernel)
        sd = {k[3:]: torch.as_tensor(g[k]) for k in g if k.startswith('sd.')}
        missing = ac.load_state_dict(sd, strict=False)
        assert [k for k in missing.missing_keys if 'extra_state' not in k] == [] and missing.unexpected_keys == []
        obs = torch.as_tensor(g['obs'], device=dev).contiguous()
        act = torch.empty((T, 4), device=dev); val = torch.empty(T, device=dev); lp = torch.empty(T, device=dev); mu = torch.empty((T, 4), device=dev)
        ac.step_into(obs, act, val, lp, mu)
        np.testing.assert_allclose(val.cpu().numpy(), g['val'], rtol=tol, atol=tol)
        eps = (torch.as_tensor(g['act'], device=dev) - mu) / torch.exp(ac.log_std)          # the reference's draws
        lp_ref = (-0.5 * eps ** 2 - ac.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        np.testing.assert_allclose(lp_ref.cpu().numpy(), g['logp'], rtol=2e-4, atol=2e-4)
        last_val = ac.value(next_obs)
    # ---- GAE with roll_out's boundaries: terminated -> 0, epoch cut -> V(next obs)
    c = lambda x: torch.as_tensor(np.asarray(x), device=dev)[:, None].contiguous()
    adv, tv, dr = compute_gae(c(g['rew']), c(g['val']), c(done), torch.zeros((T, 1), device=dev), last_val, 0.99, 0.95,
                              torch.as_tensor(g['sd.ret_oms.std'], device=dev))
    np.testing.assert_allclose(adv[:, 0].cpu().numpy(), g['adv'], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(tv[:, 0].cpu().numpy(), g['target_v'], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(dr[:, 0].cpu().numpy(), g['discounted_ret'], rtol=2e-4, atol=2e-4)
