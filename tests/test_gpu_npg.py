"""NPG / TRPO on the GPU: pdx_ppo_pi_fvp against float64 autograd's double backward, the unclipped surrogate of
pdx_ppo_pi_grad against float64 autograd, the whole NPG / TRPO / IWPG update on update_kernel='cuda' against 'torch',
and NPG / TRPO learning to hover.

Per-tensor metric, as in test_gpu_ppo_update.py: ||x - x64||_inf / ||x64||_inf <= max(4 x the same error of torch
float32 autograd on the same inputs, 1e-6)."""
import copy
import ctypes as C
import math

import pytest
import torch

from phoenix_drone_simulation_b200 import lib as _lib
from phoenix_drone_simulation_b200.npg import KL_SCALE, NPG
from phoenix_drone_simulation_b200.ppo import (PPO, _prepare, flat_views, pi_flat_params, pi_fvp, pi_fvp_torch,
                                               pi_loss_and_grad, pi_net_params)
from phoenix_drone_simulation_b200.rollout import ActorCritic
from phoenix_drone_simulation_b200.trpo import TRPO

pytestmark = pytest.mark.gpu
DEV = 'cuda'
CASES = [(1, 34, (50, 50)), (127, 34, (50, 50)), (128, 34, (50, 50)), (129, 34, (50, 50)), (5000, 34, (50, 50)),
         (262181, 34, (50, 50)), (5000, 37, (64, 64)), (5000, 160, (50, 50)), (5000, 384, (64, 64)),
         (129, 37, (7, 33)), (262181, 384, (7, 33)), (5000, 34, (64, 64)), (127, 160, (7, 33))]


def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _check(got, ref32, ref64, params, what):
    for k, (g, r32, r64) in enumerate(zip(*(flat_views(t, params) for t in (got, ref32, ref64)))):
        e, e32 = _rel(g, r64), _rel(r32, r64)
        assert e <= max(4 * e32, 1e-6), f'{what}: tensor {k} error {e:.3g} vs torch float32 {e32:.3g}'


def _case(n, obs_dim, hidden, seed, indexed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    torch.manual_seed(seed)
    ac = ActorCritic(obs_dim, pi_hidden=hidden, v_hidden=hidden, device=DEV)
    ac.set_log_std(0.7)
    rows = n + 1000 if indexed else n
    obs = torch.randn((rows, obs_dim), device=DEV, generator=g)
    idx = torch.randperm(rows, device=DEV, generator=g)[:n] if indexed else None
    v = torch.randn(pi_flat_params(ac).numel(), device=DEV, generator=g)
    return ac, obs, idx, v


@pytest.mark.parametrize('n,obs_dim,hidden', CASES)
@pytest.mark.parametrize('indexed', [False, True])
def test_fvp_matches_float64_double_backward(n, obs_dim, hidden, indexed):
    ac, obs, idx, v = _case(n, obs_dim, hidden, seed=3 * n + obs_dim, indexed=indexed)
    ac64 = copy.deepcopy(ac).double()
    params = pi_net_params(ac)
    for scale in (1.0, 0.25):
        for damping in (0.0, 0.1):
            ref64 = pi_fvp_torch(ac64, obs.double(), v.double(), damping, scale, index=idx).detach()
            ref32 = pi_fvp_torch(ac, obs, v, damping, scale, index=idx).detach()
            got = pi_fvp(ac, obs, v, damping, scale, index=idx)
            _check(got, ref32, ref64, params, f'fvp n={n} D={obs_dim} h={hidden} index={indexed} scale={scale} '
                                              f'damping={damping}')


def test_flat_views_equal_per_tensor_tensors_and_launches_are_bit_identical():
    ac, obs, idx, v = _case(262181, 34, (50, 50), seed=5, indexed=True)
    params = pi_net_params(ac)
    flat = [pi_fvp(ac, obs, v, 0.1, KL_SCALE, index=idx).clone() for _ in range(2)]
    assert torch.equal(flat[0], flat[1])
    # the same product through six separate tensors
    L, b, mlp, scratch, st = _prepare(ac, ac.pi, 4, obs, idx)
    dirs = [t.clone() for t in flat_views(v, params)]
    outs = [torch.empty_like(t) for t in dirs]
    d, g = _lib.PdxMlp(), _lib.PdxMlpGrad()
    d.hidden[0], d.hidden[1], d.n_out = 50, 50, 4
    for k in range(3):
        d.weight[k], d.bias[k] = dirs[2 * k].data_ptr(), dirs[2 * k + 1].data_ptr()
        g.weight[k], g.bias[k] = outs[2 * k].data_ptr(), outs[2 * k + 1].data_ptr()
    _lib.check(L.pdx_ppo_pi_fvp(C.byref(b), C.byref(mlp), C.c_void_p(ac.log_std.data.data_ptr()), C.byref(d),
                                KL_SCALE, 0.1, C.byref(g), C.c_void_p(scratch.data_ptr()), scratch.numel(), st))
    assert torch.equal(torch.cat([t.reshape(-1) for t in outs]), flat[0])


def _unclipped_case(n, obs_dim, hidden, seed, log_ratio_spread):
    g = torch.Generator(device=DEV).manual_seed(seed)
    torch.manual_seed(seed)
    ac = ActorCritic(obs_dim, pi_hidden=hidden, v_hidden=hidden, device=DEV)
    ac.set_log_std(0.7)
    obs = torch.randn((n, obs_dim), device=DEV, generator=g)
    with torch.no_grad():
        mu = ac.pi(obs)
        act = mu + torch.exp(ac.log_std) * torch.randn((n, 4), device=DEV, generator=g)
        logp = (-0.5 * ((act - mu) / torch.exp(ac.log_std)) ** 2 - ac.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        logp_old = logp - log_ratio_spread * (2 * torch.rand(n, device=DEV, generator=g) - 1)
    adv = torch.randn(n, device=DEV, generator=g)
    return ac, obs, act, adv, logp_old


def _unclipped_loss(pi, log_std, obs, act, adv, logp_old):
    mu = pi(obs)
    std = torch.exp(log_std)
    logp = (-0.5 * ((act - mu) / std) ** 2 - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
    return -(torch.exp(logp - logp_old) * adv).mean()


def _ref(ac, args, dtype):
    net = copy.deepcopy(ac.pi).to(dtype)
    loss = _unclipped_loss(net, ac.log_std.to(dtype), *(t.to(dtype) for t in args))
    loss.backward()
    lins = [m for m in net if isinstance(m, torch.nn.Linear)]
    return loss.detach().double(), torch.cat([p.grad.reshape(-1) for m in lins for p in (m.weight, m.bias)])


@pytest.mark.parametrize('n,obs_dim,hidden', [(129, 34, (50, 50)), (262181, 34, (50, 50)), (5000, 384, (64, 64)),
                                              (5000, 37, (7, 33))])
def test_unclipped_surrogate_matches_float64_autograd(n, obs_dim, hidden):
    ac, *args = _unclipped_case(n, obs_dim, hidden, seed=n, log_ratio_spread=2.0)   # ratios in [e^-2, e^2]
    l64, g64 = _ref(ac, args, torch.float64)
    l32, g32 = _ref(ac, args, torch.float32)
    loss, _ = pi_loss_and_grad(ac, *args, None)
    e, e32 = _rel(loss, l64), _rel(l32, l64)
    assert e <= max(4 * e32, 1e-6), (e, e32)
    got = torch.cat([p.grad.reshape(-1) for p in pi_net_params(ac)])
    _check(got, g32, g64, pi_net_params(ac), f'unclipped n={n} D={obs_dim} h={hidden}')


@pytest.mark.parametrize('spread', [60.0, 100.0])
def test_unclipped_loss_is_non_finite_exactly_when_torch_float32_is(spread):
    """exp overflows float32 beyond a log-ratio of ~88.7: spread 100 puts some ratios past it, spread 60 none (and keeps the float32 sum finite)."""
    ac, *args = _unclipped_case(5000, 34, (50, 50), seed=17, log_ratio_spread=spread)
    with torch.no_grad():
        l32 = _unclipped_loss(ac.pi, ac.log_std, *args)
    loss, _ = pi_loss_and_grad(ac, *args, None, grad=False)
    assert math.isfinite(float(loss)) == math.isfinite(float(l32)), (float(loss), float(l32))
    assert math.isfinite(float(l32)) == (spread == 60.0)


# max over parameters of max |p_cuda - p_torch| / max |p_torch - p0| after one update, measured on a B200: NPG and
# TRPO 2.5e-6 (one step, the CG solve in float32 on both paths), IWPG 0.154 (80 Adam steps on the unclipped surrogate
# amplify last-bit gradient differences more than PPO's clipped 80, measured 0.064 there)
UPDATE_BOUND = {'npg': 1e-4, 'trpo': 1e-4, 'iwpg': 0.25}


def _two(kind):
    mk = {'npg': lambda k: NPG('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=10, seed=1, update_kernel=k),
          'trpo': lambda k: TRPO('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=10, seed=1, update_kernel=k),
          'iwpg': lambda k: PPO('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=10, seed=1, update_kernel=k,
                                clip_ratio=None)}[kind]
    algs = [mk(k) for k in ('torch', 'cuda')]
    data = algs[0].collector.collect()
    return algs, data


@pytest.mark.parametrize('kind', ['npg', 'trpo', 'iwpg'])
def test_whole_update_matches_the_torch_update(kind):
    (a_t, a_c), data = _two(kind)
    infos, p0 = [], [p.detach().clone() for p in a_t.ac.parameters()]
    for a in (a_t, a_c):
        torch.manual_seed(123)                               # the same value mini-batches on both paths
        infos.append(a.update(data))
    info_t, info_c = infos
    worst = 0.0
    for (name, pt), pc, q0 in zip(a_t.ac.named_parameters(), a_c.ac.parameters(), p0):
        change = float((pt.detach() - q0).abs().max())
        if change == 0.0:
            assert torch.equal(pt, pc), name
            continue
        worst = max(worst, float((pt.detach() - pc.detach()).abs().max()) / change)
    print(f'{kind}: max |p_cuda - p_torch| / max |p_torch - p0| = {worst:.3g}; torch {info_t}; cuda {info_c}')
    assert worst < UPDATE_BOUND[kind], (kind, worst)
    if kind != 'iwpg':
        assert info_t['accept_step'] == info_c['accept_step']
        assert abs(info_t['xHx'] - info_c['xHx']) <= 1e-3 * abs(info_t['xHx'])
        if kind == 'trpo' and info_c['accept_step'] > 0:
            for info in (info_t, info_c):
                assert 0 < info['kl'] <= 1.5 * a_c.target_kl
        if kind == 'npg':
            assert info_c['accept_step'] == 1


EPOCHS = {'npg': 12, 'trpo': 12}


@pytest.mark.parametrize('kind', ['npg', 'trpo'])
def test_learns_to_hover_with_the_cuda_update(kind):
    """The thresholds of test_gpu_collector.test_ppo_learns_to_hover with update_kernel='cuda'.  Observed on a B200
    (episodes, EpLen) per epoch, the same for NPG and TRPO (every line search accepted its first candidate):
    (29133, 8.1) (19623, 12.5) (18732, 13.9) (14653, 16.9) (8320, 25.4) (4400, 45.9) (3244, 70.0) (3036, 85.4)
    (3039, 86.8) (3327, 83.6) (3745, 76.1) (3903, 68.6)."""
    cls = {'npg': NPG, 'trpo': TRPO}[kind]
    alg = cls('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=EPOCHS[kind], seed=0, update_kernel='cuda')
    alg.learn()
    print(kind, [(r['episodes'], round(r['EpLen'], 1), r['accept_step']) for r in alg.history])
    first, last = alg.history[0], alg.history[-1]
    assert all(math.isfinite(r['loss_v']) and math.isfinite(r['loss_pi']) for r in alg.history)
    assert last['episodes'] < 0.25 * first['episodes'], (first, last)
    assert last['EpLen'] > 2 * first['EpLen']
