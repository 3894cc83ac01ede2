"""The fused PPO update kernels (pdx_ppo_pi_grad / pdx_ppo_v_grad) against float64 autograd, and PPO(update_kernel=
'cuda') against the torch update it replaces.

Gradient metric, per parameter: ||g - g64||_inf / ||g64||_inf must be <= max(4 x the same error of torch float32
autograd on the same inputs, 1e-6).  The losses are held to the same rule."""
import copy
import math

import pytest
import torch

from phoenix_drone_simulation_b200.ppo import PPO, pi_loss_and_grad, v_loss_and_grad
from phoenix_drone_simulation_b200.rollout import ActorCritic

pytestmark = pytest.mark.gpu
DEV = 'cuda'
CLIP = 0.2


def _lins(net):
    return [m for m in net if isinstance(m, torch.nn.Linear)]


def _params(net):
    return [p for lin in _lins(net) for p in (lin.weight, lin.bias)]


def _pi_loss(pi, log_std, obs, act, adv, logp_old):
    """PPO._loss_pi without the entropy term."""
    mu = pi(obs)
    std = torch.exp(log_std)
    logp = (-0.5 * ((act - mu) / std) ** 2 - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
    ratio = torch.exp(logp - logp_old)
    return -torch.min(ratio * adv, adv * torch.clamp(ratio, 1 - CLIP, 1 + CLIP)).mean()


def _ref_grads(net, loss_fn, dtype):
    n = copy.deepcopy(net).to(dtype)
    for p in n.parameters():
        p.grad = None
    loss = loss_fn(n)
    loss.backward()
    return loss.detach().double(), [p.grad.double() for p in _params(n)]


def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _check(loss, grads, ref32, ref64, what):
    worst = []
    for k, (g, g32, g64) in enumerate(zip([loss] + grads, [ref32[0]] + ref32[1], [ref64[0]] + ref64[1])):
        e, e32 = _rel(g, g64), _rel(g32, g64)
        assert e <= max(4 * e32, 1e-6), f'{what}: tensor {k} (0 = loss) error {e:.3g} vs torch float32 {e32:.3g}'
        worst.append(e)
    return max(worst)


def _actor_case(n, obs_dim, hidden, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    torch.manual_seed(seed)
    ac = ActorCritic(obs_dim, pi_hidden=hidden, v_hidden=hidden, device=DEV)
    ac.set_log_std(0.7)
    obs = torch.randn((n, obs_dim), device=DEV, generator=g)
    with torch.no_grad():
        pi64 = copy.deepcopy(ac.pi).double()
        mu64 = pi64(obs.double())
        ls64 = ac.log_std.double()
        act = (mu64 + torch.exp(ls64) * torch.randn((n, 4), device=DEV, generator=g, dtype=torch.float64)).float()
        logp64 = (-0.5 * ((act.double() - mu64) / torch.exp(ls64)) ** 2 - ls64 - 0.5 * math.log(2 * math.pi)).sum(-1)
        # target ratios on both sides of both clip bounds, never within 1e-3 of 1 +- CLIP
        u = torch.rand(n, device=DEV, generator=g, dtype=torch.float64)
        lo, hi = 1 - CLIP, 1 + CLIP
        r = torch.where(u < 0.3, lo - 0.001 - 0.3 * u, torch.where(u < 0.7, lo + 0.001 + (u - 0.3) / 0.4 * (hi - lo - 0.002),
                                                                    hi + 0.001 + (u - 0.7)))
        logp_old = (logp64 - torch.log(r)).float()
        r_true = torch.exp(logp64 - logp_old.double())
        assert float(torch.minimum((r_true - lo).abs(), (r_true - hi).abs()).min()) > 1e-4
        adv = torch.randn(n, device=DEV, generator=g)
    return ac, obs, act, adv, logp_old


CASES = [(1, 34, (50, 50)), (127, 34, (50, 50)), (128, 34, (50, 50)), (129, 34, (50, 50)), (5000, 34, (50, 50)),
         (262181, 34, (50, 50)), (5000, 37, (64, 64)), (5000, 160, (50, 50)), (5000, 384, (64, 64)),
         (129, 37, (7, 33)), (262181, 384, (7, 33)), (5000, 34, (64, 64)), (127, 160, (7, 33))]


@pytest.mark.parametrize('n,obs_dim,hidden', CASES)
def test_actor_gradients_match_float64_autograd(n, obs_dim, hidden):
    ac, obs, act, adv, logp_old = _actor_case(n, obs_dim, hidden, seed=n + obs_dim)
    with torch.no_grad():   # both clip sides are populated where the batch is large enough
        mu = ac.pi(obs)
        r = torch.exp((-0.5 * ((act - mu) / torch.exp(ac.log_std)) ** 2 - ac.log_std).sum(-1)
                      - 2 * math.log(2 * math.pi) - logp_old)
        if n >= 5000:
            assert int((r < 1 - CLIP).sum()) > n // 10 and int((r > 1 + CLIP).sum()) > n // 10
    fn = lambda dt: (lambda net: _pi_loss(net, ac.log_std.to(dt), obs.to(dt), act.to(dt), adv.to(dt), logp_old.to(dt)))
    ref64, ref32 = _ref_grads(ac.pi, fn(torch.float64), torch.float64), _ref_grads(ac.pi, fn(torch.float32), torch.float32)
    loss, kl = pi_loss_and_grad(ac, obs, act, adv, logp_old, CLIP)
    assert kl is None and ac.log_std.grad is None
    _check(loss, [p.grad for p in _params(ac.pi)], ref32, ref64, f'actor n={n} D={obs_dim} h={hidden}')


@pytest.mark.parametrize('n,obs_dim,hidden', CASES)
@pytest.mark.parametrize('indexed', [False, True])
def test_critic_gradients_match_float64_autograd(n, obs_dim, hidden, indexed):
    g = torch.Generator(device=DEV).manual_seed(7 * n + obs_dim)
    torch.manual_seed(n)
    ac = ActorCritic(obs_dim, pi_hidden=hidden, v_hidden=hidden, device=DEV)
    rows = n + 1000 if indexed else n
    obs = torch.randn((rows, obs_dim), device=DEV, generator=g)
    target = torch.randn(rows, device=DEV, generator=g)
    idx = torch.randperm(rows, device=DEV, generator=g)[:n] if indexed else None
    o, t = (obs[idx], target[idx]) if indexed else (obs, target)
    fn = lambda dt: (lambda net: ((net(o.to(dt)).squeeze(-1) - t.to(dt)) ** 2).mean())
    ref64, ref32 = _ref_grads(ac.v, fn(torch.float64), torch.float64), _ref_grads(ac.v, fn(torch.float32), torch.float32)
    loss = v_loss_and_grad(ac, obs, target, idx)
    _check(loss, [p.grad for p in _params(ac.v)], ref32, ref64, f'critic n={n} D={obs_dim} h={hidden} index={indexed}')


@pytest.mark.parametrize('n,obs_dim,hidden', [(129, 34, (50, 50)), (5000, 384, (64, 64)), (262181, 34, (50, 50))])
def test_forward_only_mode_gives_mu_and_kl(n, obs_dim, hidden):
    ac, obs, act, adv, logp_old = _actor_case(n, obs_dim, hidden, seed=3)
    mu = torch.empty((n, 4), device=DEV)
    with torch.no_grad():
        mu_ref = ac.pi(obs) + 0.05 * torch.randn((n, 4), device=DEV)
    for p in _params(ac.pi):
        p.grad = None
    loss, kl = pi_loss_and_grad(ac, obs, act, adv, logp_old, CLIP, grad=False, mu=mu, mu_ref=mu_ref)
    assert all(p.grad is None for p in _params(ac.pi))
    with torch.no_grad():
        torch.testing.assert_close(mu, ac.pi(obs), rtol=1e-5, atol=1e-6)
        # the expression of PPO.update (log_std frozen: std_n == std_old)
        std = torch.exp(ac.log_std)
        k32 = (torch.log(std / std) + (std ** 2 + (mu_ref - mu) ** 2) / (2 * std ** 2) - 0.5).sum(-1).mean()
        k64 = (((mu_ref.double() - copy.deepcopy(ac.pi).double()(obs.double())) ** 2) / (2 * std.double() ** 2)).sum(-1).mean()
        assert abs(float(kl) - float(k64)) <= 1e-5 * abs(float(k64)), (float(kl), float(k64))
        assert abs(float(kl) - float(k32)) <= 1e-3 * abs(float(k64)), (float(kl), float(k32))
        l32 = _pi_loss(ac.pi, ac.log_std, obs, act, adv, logp_old)
        assert abs(float(loss) - float(l32)) <= 1e-5 * abs(float(l32)) + 1e-7


def test_two_launches_are_bit_identical():
    ac, obs, act, adv, logp_old = _actor_case(262181, 34, (50, 50), seed=11)
    out = []
    for _ in range(2):
        loss, _ = pi_loss_and_grad(ac, obs, act, adv, logp_old, CLIP)
        vloss = v_loss_and_grad(ac, obs, adv, torch.arange(100000, 200000, device=DEV))
        out.append([loss.clone(), vloss.clone()] + [p.grad.clone() for p in _params(ac.pi) + _params(ac.v)])
    for a, b in zip(*out):
        assert torch.equal(a, b)


def _two_ppos(**kw):
    algs = [PPO('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=10, seed=1, update_kernel=k, **kw)
            for k in ('torch', 'cuda')]
    data = algs[0].collector.collect()
    for (name, p), q in zip(algs[0].ac.named_parameters(), algs[1].ac.parameters()):
        assert torch.equal(p, q), name
    return algs, data


def _update(alg, data):
    torch.manual_seed(123)                                   # the same mini-batch permutations for both paths
    p0 = [p.detach().clone() for p in alg.ac.parameters()]
    info = alg.update(data)
    return info, p0


# max over parameters of max |p_cuda - p_torch| / max |p_torch - p0| after one update of 80 + 80 steps (Adam amplifies
# last-bit gradient differences of near-zero entries); measured 0.064 on a B200
UPDATE_BOUND = 0.1


def test_whole_update_matches_the_torch_update():
    (a_t, a_c), data = _two_ppos()
    info_t, p0 = _update(a_t, data)
    info_c, _ = _update(a_c, data)
    assert info_t['pi_iters'] == info_c['pi_iters'] == 80
    worst = 0.0
    for (name, pt), pc, q0 in zip(a_t.ac.named_parameters(), a_c.ac.parameters(), p0):
        change = float((pt - q0).abs().max())
        if change == 0.0:                                    # log_std, normaliser
            assert torch.equal(pt, pc), name
            continue
        frac = float((pt - pc).abs().max()) / change
        worst = max(worst, frac)
        assert frac < UPDATE_BOUND, (name, frac)
    print(f'whole update: max |p_cuda - p_torch| / max |p_torch - p0| = {worst:.3g}')
    assert abs(info_t['loss_pi'] - info_c['loss_pi']) <= 1e-3 * float(data['adv'].abs().mean())
    assert abs(info_t['loss_v'] - info_c['loss_v']) <= 1e-3 * abs(info_t['loss_v'])


def test_kl_early_stopping_stops_at_the_same_iteration():
    (a_t, a_c), data = _two_ppos(use_kl_early_stopping=True, target_kl=1e9)
    probe = copy.deepcopy(a_t.ac.state_dict())
    kl_full = _update(a_t, data)[0]['kl']                   # the KL after all 80 iterations
    a_t.ac.load_state_dict(probe)
    a_t.pi_opt = torch.optim.Adam(a_t.ac.pi.parameters(), lr=3e-4)
    a_t.vf_opt = torch.optim.Adam(a_t.ac.v.parameters(), lr=1e-3)
    for a in (a_t, a_c):
        a.target_kl = kl_full / 4
    info_t, info_c = _update(a_t, data)[0], _update(a_c, data)[0]
    print(f"kl early stopping: target {kl_full / 4:.3g}, pi_iters torch {info_t['pi_iters']} cuda {info_c['pi_iters']}")
    assert 1 < info_t['pi_iters'] < 80
    assert info_t['pi_iters'] == info_c['pi_iters']


def test_ppo_with_cuda_update_learns_to_hover():
    """The thresholds of test_gpu_collector.test_ppo_learns_to_hover with update_kernel='cuda'."""
    alg = PPO('DroneHoverSimpleEnv-v0', num_envs=4096, steps=64, epochs=12, seed=0, update_kernel='cuda')
    alg.learn()
    first, last = alg.history[0], alg.history[-1]
    assert all(math.isfinite(r['loss_v']) and math.isfinite(r['loss_pi']) for r in alg.history)
    assert last['episodes'] < 0.25 * first['episodes'], (first, last)
    assert last['EpLen'] > 2 * first['EpLen']
