"""PopulationPPO and its member kernels against the single-agent pieces they are built from.

Every member kernel must equal its single-network sibling on the member's slice bit for bit (the moments to 1e-12
relative: float64 sums in another order); a population rollout must equal single-agent rollouts over VecEnv(num_envs=N,
env_offset=m N); a population update must equal single-agent PPO updates given the same data and permutations."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch

from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.policy_io import evaluate_many
from phoenix_drone_simulation_b200.population import PopulationPPO
from phoenix_drone_simulation_b200.ppo import PPO, pi_loss_and_grad, v_loss_and_grad
from phoenix_drone_simulation_b200.rollout import ActorCritic, RolloutCollector, column_moments, compute_gae
from phoenix_drone_simulation_b200.vec_env import VecEnv

pytestmark = pytest.mark.gpu
DEV = 'cuda'
ENV = 'DroneHoverSimpleEnv-v0'


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _lins(net):
    return [m for m in net if isinstance(m, torch.nn.Linear)]


def _members(P, obs_dim, hidden, seed, norm=True):
    """P ActorCritics with random weights, log_std and normalisers."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    acs = []
    for m in range(P):
        torch.manual_seed(seed + m)
        ac = ActorCritic(obs_dim, pi_hidden=hidden, v_hidden=(64, 64), device=DEV, policy_kernel='cuda',
                         use_standardized_obs=norm)
        with torch.no_grad():
            ac.set_log_std(0.3 + 0.2 * m)
            if norm:
                ac.obs_oms.mean.copy_(0.3 * torch.randn(obs_dim, device=DEV, generator=g))
                ac.obs_oms.std.copy_(0.5 + torch.rand(obs_dim, device=DEV, generator=g))
        acs.append(ac)
    return acs


def _mlp(params, n_out):
    st = L.PdxMlp()
    st.hidden[0], st.hidden[1], st.n_out = params[0].shape[-2], params[2].shape[-2], n_out
    for k in range(3):
        st.weight[k], st.bias[k] = params[2 * k].data_ptr(), params[2 * k + 1].data_ptr()
    return st


# ---- 1. policy step -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('P', [1, 3, 7])
@pytest.mark.parametrize('hidden', [(50, 50), (64, 64)])
@pytest.mark.parametrize('norm', [True, False])
def test_policy_step_members_equals_single(P, hidden, norm):
    lib = L.load()
    N, D, offset, seed, counter = 1000, 34, 12345, 77, 5
    acs = _members(P, D, hidden, seed=P * 10 + hidden[0], norm=norm)
    pi0, v0 = acs[0]._mlp_struct(acs[0].pi, 4), acs[0]._mlp_struct(acs[0].v, 1)
    words = int(lib.pdx_policy_pack_words(D, C.byref(pi0), C.byref(v0)))
    stride = words + 8                                        # images need not be packed back to back
    packed = torch.zeros((P, stride), dtype=torch.float32, device=DEV)
    for m, ac in enumerate(acs):
        pi, v = ac._mlp_struct(ac.pi, 4), ac._mlp_struct(ac.v, 1)
        L.check(lib.pdx_policy_pack(D, C.byref(pi), C.byref(v), _p(packed[m]), _st()))
    obs = torch.randn((P, N, D), device=DEV, generator=torch.Generator(device=DEV).manual_seed(P))
    mean = torch.stack([ac.obs_oms.mean for ac in acs]).contiguous() if norm else None
    std = torch.stack([ac.obs_oms.std for ac in acs]).contiguous() if norm else None
    log_std = torch.stack([ac.log_std for ac in acs]).contiguous()
    out = [torch.full(s, float('nan'), device=DEV) for s in ((P, N, 4), (P, N), (P, N), (P, N, 4))]
    L.check(lib.pdx_policy_step_members(P, N, D, _p(obs), _p(mean), _p(std), 1e-5, C.byref(pi0), C.byref(v0),
                                        _p(log_std), _p(packed), stride, seed, counter, offset, *map(_p, out), _st()))
    for m, ac in enumerate(acs):
        ref = [torch.full_like(o[m], float('nan')) for o in out]
        pi, v = ac._mlp_struct(ac.pi, 4), ac._mlp_struct(ac.v, 1)
        L.check(lib.pdx_policy_step(N, D, _p(obs[m]), _p(mean[m] if norm else None), _p(std[m] if norm else None), 1e-5,
                                    C.byref(pi), C.byref(v), _p(ac.log_std.data), _p(packed[m]), seed, counter,
                                    offset + m * N, *map(_p, ref), _st()))
        for name, a, b in zip(('act', 'val', 'logp', 'mu'), out, ref):
            assert torch.equal(a[m], b), (m, name)


# ---- 2. losses and gradients ---------------------------------------------------------------------------------------
def _ppo_case(P, n, rows, D, seed, hidden=(50, 50)):
    acs = _members(P, D, hidden, seed)
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.randn((P, rows, D), device=DEV, generator=g)
    act = torch.randn((P, rows, 4), device=DEV, generator=g)
    adv = torch.randn((P, rows), device=DEV, generator=g)
    logp_old = -4 + 0.5 * torch.randn((P, rows), device=DEV, generator=g)
    target_v = torch.randn((P, rows), device=DEV, generator=g)
    return acs, obs, act, adv, logp_old, target_v


def _scratch(ac, net, n_out, D):
    mlp = ac._mlp_struct(net, n_out)
    return int(L.load().pdx_ppo_scratch_bytes(0, D, C.byref(mlp)))


@pytest.mark.parametrize('clip', [0.2, None])
@pytest.mark.parametrize('indexed', [False, True])
@pytest.mark.parametrize('hidden', [(50, 50), (64, 64)])
@pytest.mark.parametrize('n,D', [(1, 34), (300, 34), (148 * 128 + 77, 34), (2000, 384)])
def test_pi_grad_members_equals_single(clip, indexed, hidden, n, D):
    P = 3
    rows = n + 13 if indexed else n
    acs, obs, act, adv, logp_old, _ = _ppo_case(P, n, rows, D, seed=n + D, hidden=hidden)
    idx = torch.stack([torch.randperm(rows, device=DEV)[:n] for _ in range(P)]).contiguous() if indexed else None
    pis = [torch.stack([getattr(_lins(ac.pi)[k], a).detach() for ac in acs]).contiguous()
           for k in range(3) for a in ('weight', 'bias')]
    grads = [torch.full_like(t, float('nan')) for t in pis]
    gs = L.PdxMlpGrad()
    for k in range(3):
        gs.weight[k], gs.bias[k] = grads[2 * k].data_ptr(), grads[2 * k + 1].data_ptr()
    log_std = torch.stack([ac.log_std for ac in acs]).contiguous()
    mu_ref = torch.randn((P, n, 4), device=DEV)
    mu = torch.empty((P, n, 4), device=DEV)
    loss, kl = torch.empty(P, device=DEV), torch.empty(P, device=DEV)
    per = _scratch(acs[0], acs[0].pi, 4, D)
    scratch = torch.empty(P * per, dtype=torch.uint8, device=DEV)
    b = L.PdxPpoBatch()
    b.n, b.obs_dim, b.obs, b.index = n, D, obs.data_ptr(), idx.data_ptr() if indexed else None
    b.act, b.adv, b.logp_old = act.data_ptr(), adv.data_ptr(), logp_old.data_ptr()
    clip_v = math.inf if clip is None else clip
    L.check(L.load().pdx_ppo_pi_grad_members(P, C.byref(b), rows, None, C.byref(_mlp(pis, 4)), _p(log_std), clip_v,
                                             C.byref(gs), _p(loss), _p(mu), _p(mu_ref), _p(kl), _p(scratch),
                                             scratch.numel(), _st()))
    for m, ac in enumerate(acs):
        mu1 = torch.empty((n, 4), device=DEV)
        l1, k1 = pi_loss_and_grad(ac, obs[m].contiguous(), act[m].contiguous(), adv[m].contiguous(),
                                  logp_old[m].contiguous(), clip, index=idx[m].contiguous() if indexed else None,
                                  mu=mu1, mu_ref=mu_ref[m].contiguous())
        assert torch.equal(loss[m], l1) and torch.equal(kl[m], k1), m
        assert torch.equal(mu[m], mu1), m
        ref = [p_.grad for lin in _lins(ac.pi) for p_ in (lin.weight, lin.bias)]
        for j, (a, r) in enumerate(zip(grads, ref)):
            assert torch.equal(a[m], r), (m, j)
    if n == 300 and not indexed and clip is not None:             # and against float64 autograd, like the single kernel
        m = 1
        pi64 = copy.deepcopy(acs[m].pi).double()
        o, a_, ad, lo = obs[m].double(), act[m].double(), adv[m].double(), logp_old[m].double()
        ls = acs[m].log_std.double()
        mu64 = pi64(o)
        logp = (-0.5 * ((a_ - mu64) / torch.exp(ls)) ** 2 - ls - 0.5 * math.log(2 * math.pi)).sum(-1)
        r = torch.exp(logp - lo)
        l64 = -torch.min(r * ad, ad * torch.clamp(r, 1 - clip, 1 + clip)).mean()
        l64.backward()
        for j, p64 in enumerate(p_ for lin in _lins(pi64) for p_ in (lin.weight, lin.bias)):
            err = float((grads[j][m].double() - p64.grad).abs().max() / p64.grad.abs().max())
            assert err < 1e-4, (j, err)
        assert abs(float(loss[m]) - float(l64.detach())) <= 1e-5 * max(1.0, abs(float(l64.detach())))


@pytest.mark.parametrize('n,D', [(1, 34), (2048, 34), (148 * 128 + 77, 34), (2000, 384)])
def test_v_grad_members_equals_single(n, D):
    P, rows = 4, n + 100
    acs, obs, _, _, _, target_v = _ppo_case(P, n, rows, D, seed=n * 3 + D)
    idx = torch.stack([torch.randperm(rows, device=DEV)[:n] for _ in range(P)]).contiguous()
    vs = [torch.stack([getattr(_lins(ac.v)[k], a).detach() for ac in acs]).contiguous()
          for k in range(3) for a in ('weight', 'bias')]
    grads = [torch.full_like(t, float('nan')) for t in vs]
    gs = L.PdxMlpGrad()
    for k in range(3):
        gs.weight[k], gs.bias[k] = grads[2 * k].data_ptr(), grads[2 * k + 1].data_ptr()
    loss = torch.empty(P, device=DEV)
    per = _scratch(acs[0], acs[0].v, 1, D)
    scratch = torch.empty(P * per, dtype=torch.uint8, device=DEV)
    b = L.PdxPpoBatch()
    b.n, b.obs_dim, b.obs, b.index, b.target_v = n, D, obs.data_ptr(), idx.data_ptr(), target_v.data_ptr()
    L.check(L.load().pdx_ppo_v_grad_members(P, C.byref(b), rows, None, C.byref(_mlp(vs, 1)), C.byref(gs), _p(loss),
                                            _p(scratch), scratch.numel(), _st()))
    for m, ac in enumerate(acs):
        l1 = v_loss_and_grad(ac, obs[m].contiguous(), target_v[m].contiguous(), idx[m].contiguous())
        assert torch.equal(loss[m], l1), m
        ref = [p_.grad for lin in _lins(ac.v) for p_ in (lin.weight, lin.bias)]
        for j, (a, r) in enumerate(zip(grads, ref)):
            assert torch.equal(a[m], r), (m, j)


def test_pi_grad_members_active_mask_leaves_inactive_members_alone():
    P, n, D = 4, 5000, 34
    acs, obs, act, adv, logp_old, _ = _ppo_case(P, n, n, D, seed=5)
    pis = [torch.stack([getattr(_lins(ac.pi)[k], a).detach() for ac in acs]).contiguous()
           for k in range(3) for a in ('weight', 'bias')]
    grads = [torch.full_like(t, 7.0) for t in pis]
    gs = L.PdxMlpGrad()
    for k in range(3):
        gs.weight[k], gs.bias[k] = grads[2 * k].data_ptr(), grads[2 * k + 1].data_ptr()
    log_std = torch.stack([ac.log_std for ac in acs]).contiguous()
    mu_ref = torch.randn((P, n, 4), device=DEV)
    mu = torch.full((P, n, 4), 7.0, device=DEV)
    loss, kl = torch.full((P,), 7.0, device=DEV), torch.full((P,), 7.0, device=DEV)
    active = torch.tensor([1, 0, 1, 0], dtype=torch.uint8, device=DEV)
    scratch = torch.empty(P * _scratch(acs[0], acs[0].pi, 4, D), dtype=torch.uint8, device=DEV)
    b = L.PdxPpoBatch()
    b.n, b.obs_dim, b.obs = n, D, obs.data_ptr()
    b.act, b.adv, b.logp_old = act.data_ptr(), adv.data_ptr(), logp_old.data_ptr()
    L.check(L.load().pdx_ppo_pi_grad_members(P, C.byref(b), n, _p(active), C.byref(_mlp(pis, 4)), _p(log_std), 0.2,
                                             C.byref(gs), _p(loss), _p(mu), _p(mu_ref), _p(kl), _p(scratch),
                                             scratch.numel(), _st()))
    for m, ac in enumerate(acs):
        if active[m]:
            mu1 = torch.empty((n, 4), device=DEV)
            l1, k1 = pi_loss_and_grad(ac, obs[m].contiguous(), act[m].contiguous(), adv[m].contiguous(),
                                      logp_old[m].contiguous(), 0.2, mu=mu1, mu_ref=mu_ref[m].contiguous())
            assert torch.equal(loss[m], l1) and torch.equal(kl[m], k1) and torch.equal(mu[m], mu1)
            ref = [p_.grad for lin in _lins(ac.pi) for p_ in (lin.weight, lin.bias)]
            assert all(torch.equal(a[m], r) for a, r in zip(grads, ref))
        else:
            assert float(loss[m]) == 7.0 and float(kl[m]) == 7.0 and bool((mu[m] == 7.0).all())
            assert all(bool((a[m] == 7.0).all()) for a in grads)


# ---- 3. GAE and moments --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('scaling', [True, False])
def test_gae_members_equals_single(scaling):
    P, N, T = 5, 333, 64
    g = torch.Generator(device=DEV).manual_seed(11)
    rew = torch.randn((T, P * N), device=DEV, generator=g)
    val = torch.randn((T, P * N), device=DEV, generator=g)
    boot = torch.randn((T, P * N), device=DEV, generator=g)
    last = torch.randn(P * N, device=DEV, generator=g)
    u = torch.rand((T, P * N), device=DEV, generator=g)
    done = torch.where(u < 0.03, 1, torch.where(u < 0.06, 2, 0)).to(torch.uint8)
    ret_std = (0.2 + torch.rand(P, device=DEV, generator=g)).contiguous()
    outs = [torch.empty((T, P * N), device=DEV) for _ in range(3)]
    L.check(L.load().pdx_gae_members(P, T, N, _p(rew), _p(val), _p(done), _p(boot), _p(last), 0.99, 0.95, 1e-5,
                                     1 if scaling else 0, _p(ret_std) if scaling else None, *map(_p, outs), _st()))
    for m in range(P):
        s = slice(m * N, (m + 1) * N)
        ref = compute_gae(rew[:, s].contiguous(), val[:, s].contiguous(), done[:, s].contiguous(),
                          boot[:, s].contiguous(), last[s].contiguous(), 0.99, 0.95,
                          ret_std[m:m + 1] if scaling else None)
        for a, r in zip(outs, ref):
            assert torch.equal(a[:, s], r), m


@pytest.mark.parametrize('dim,shifted', [(34, False), (34, True), (1, False), (384, True)])
def test_moments_members_match_single(dim, shifted):
    P, N, T = 3, 700, 16
    g = torch.Generator(device=DEV).manual_seed(dim)
    x = (1 + 3 * torch.randn((T, P * N, dim), device=DEV, generator=g)).contiguous()
    shift = torch.randn((P, dim), device=DEV, generator=g, dtype=torch.float64).contiguous() if shifted else None
    out = torch.zeros((P, 2 * dim), dtype=torch.float64, device=DEV)
    L.check(L.load().pdx_moments_members(P, T, N, dim, _p(x), _p(shift), _p(out), _st()))
    for m in range(P):
        s1, s2 = column_moments(x[:, m * N:(m + 1) * N], shift[m] if shifted else None)
        ref = torch.cat([s1, s2])
        assert float(((out[m] - ref).abs() / ref.abs().clamp_min(1e-300)).max()) <= 1e-12, m


# ---- 4. rollout ----------------------------------------------------------------------------------------------------
def test_population_rollout_equals_single_agents():
    P, N, T, seed = 3, 300, 48, 3
    pop = PopulationPPO(ENV, members=P, num_envs_per_member=N, steps=T, seed=seed)
    singles = [pop.member(m) for m in range(P)]
    data = pop.collect()
    stats = pop.episode_stats()
    assert not pop.reset_each_rollout
    for m in range(P):
        env = VecEnv(ENV, N, seed=seed, env_offset=m * N, keep_final_obs=True)
        col = RolloutCollector(env, singles[m], T, reset_each_rollout=False)
        ref = col.collect()
        assert not col.fused_used
        s = slice(m * N, (m + 1) * N)
        assert torch.equal(pop.obs[:, s], col.obs), m
        for k in ('act', 'log_p', 'val', 'rew', 'done', 'adv', 'target_v', 'discounted_ret'):
            assert torch.equal(data[k][:, s], ref[k]), (m, k)
        assert torch.equal(pop.boot[:, s], col.boot) and torch.equal(pop.last_val[s], col.last_val), m
        es = env.episode_stats()
        assert float(stats[m, 0]) == float(es[0]), m
        assert torch.equal(stats[m, 4:], es[4:]), m
        assert torch.allclose(stats[m, 1:4], es[1:4], rtol=1e-12, atol=0), m


# ---- 5. update -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kernel', ['torch', 'cuda'])
def test_population_update_equals_single_agents(kernel, monkeypatch):
    P, N, T, seed = 3, 512, 32, 1
    kw = dict(steps=T, seed=seed, update_kernel=kernel, use_kl_early_stopping=True, target_kl=0.002,
              train_pi_iterations=40)
    pop = PopulationPPO(ENV, members=P, num_envs_per_member=N, **kw)
    data = pop.collect()
    singles = []
    for m in range(P):
        alg = PPO(ENV, num_envs=N, **kw)
        alg.ac.load_state_dict(pop.member(m).state_dict())
        singles.append(alg)
    perms, randperm = [], torch.randperm

    def record(*a, **k):
        perms.append(randperm(*a, **k))
        return perms[-1]
    monkeypatch.setattr(torch, 'randperm', record)
    info = pop.update(data)
    for m, alg in enumerate(singles):
        replay = iter(perms[m::P])
        monkeypatch.setattr(torch, 'randperm', lambda *a, **k: next(replay))
        s = slice(m * N, (m + 1) * N)
        dm = {k: data[k][:, s] for k in ('obs', 'act', 'adv', 'target_v', 'log_p', 'rew')}
        ref = alg.update(dm)
        assert info['pi_iters'][m] == ref['pi_iters'], (m, info['pi_iters'], ref['pi_iters'])
        got = pop.member(m)
        for a, b in zip(got.parameters(), alg.ac.parameters()):
            err = float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))
            assert err <= 1e-5, (m, err)
        assert math.isclose(info['loss_v'][m], ref['loss_v'], rel_tol=1e-4, abs_tol=1e-6)
        assert math.isclose(info['loss_pi'][m], ref['loss_pi'], rel_tol=1e-4, abs_tol=1e-6)
    # KL early stopping must have exercised the per-member mask: members stopped at different iterations, and at
    # least one before the last
    assert len(set(info['pi_iters'])) > 1, info['pi_iters']
    assert min(info['pi_iters']) < kw['train_pi_iterations'], info['pi_iters']


def test_stacked_adam_matches_torch_adam_per_member():
    """Each member of StackedAdam follows torch.optim.Adam to float32 rounding; a masked member does not move."""
    from phoenix_drone_simulation_b200.population import StackedAdam
    g = torch.Generator(device=DEV).manual_seed(3)
    P = 3
    w = torch.randn((P, 50, 34), device=DEV, generator=g).requires_grad_(True)
    refs = [w[m].detach().clone().requires_grad_(True) for m in range(P)]
    opt = StackedAdam([w], P)
    ref_opts = [torch.optim.Adam([r], lr=3e-4) for r in refs]
    for it in range(30):
        grad = torch.randn((P, 50, 34), device=DEV, generator=g)
        active = torch.tensor([True, it < 10, True], device=DEV)
        w.grad = grad
        opt.step(3e-4, active)
        for m in range(P):
            if bool(active[m]):
                refs[m].grad = grad[m].clone()
                ref_opts[m].step()
    for m in range(P):
        err = float((w[m] - refs[m]).abs().max() / refs[m].abs().max())
        assert err <= 1e-6, (m, err)
    assert opt.steps.tolist() == [30.0, 10.0, 30.0]


# ---- 6. learning ---------------------------------------------------------------------------------------------------
def test_population_learns_to_hover():
    """test_ppo_with_cuda_update_learns_to_hover's thresholds for every member, and every member's mean reward per
    environment step rises.  The mean return of the finished episodes (EpRet) is not the signal on this task: a crash
    ends an episode with a -100 penalty, so the first episodes return about -102, and as a member learns to stay up its
    finished episodes get longer and collect more per-step penalty (EpRet keeps falling for at least 60 epochs at this
    size).  The reward per step counts the crashes where they happen and the per-step penalty of the steps survived."""
    P, T, N = 4, 64, 4096
    pop = PopulationPPO(ENV, members=P, num_envs_per_member=N, steps=T, epochs=12, seed=0, update_kernel='cuda')
    rate = []
    for _ in range(pop.epochs):
        pop.learn_one_epoch()
        rate.append(pop.rew.view(T, P, N).double().mean((0, 2)).tolist())   # this epoch's rollout, per member
    first, last = pop.history[0], pop.history[-1]
    assert all(all(math.isfinite(v) for v in r['loss_v'] + r['loss_pi']) for r in pop.history)
    for m in range(P):
        assert last['episodes'][m] < 0.25 * first['episodes'][m], (m, first['episodes'], last['episodes'])
        assert last['EpLen'][m] > 2 * first['EpLen'][m], (m, first['EpLen'], last['EpLen'])
        assert rate[-1][m] > 0.5 * rate[0][m], (m, rate[0], rate[-1])       # rewards are negative: less than half
    print('reward per step', rate[0], rate[-1], 'EpRet', first['EpRet'], last['EpRet'])


# ---- 7. evaluation -------------------------------------------------------------------------------------------------
def test_evaluate_many_of_members_equals_each_alone():
    pop = PopulationPPO(ENV, members=3, num_envs_per_member=256, steps=32, epochs=2, seed=4, update_kernel='cuda')
    pop.learn()
    acs = [pop.member(m) for m in range(3)]
    together = evaluate_many(ENV, acs, 64, seed=9)
    for m, ac in enumerate(acs):
        alone = evaluate_many(ENV, [ac], 64, seed=9)
        for a, b in zip(together, alone):
            np.testing.assert_array_equal(a[m], b[0])
