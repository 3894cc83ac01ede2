"""PPO on the batched engine: rollouts by the device-side collector, update in torch or in fused CUDA kernels.

Mirrors the reference's on-policy loop (paths relative to phoenix_drone_simulation/):
  algs/iwpg/iwpg.py:259-326  learn / learn_one_epoch (roll_out -> update -> log), linear learning
                             rate decay (:208-221), exploration-noise annealing (:272-273)
  algs/iwpg/iwpg.py:398-485  update(): value net `train_v_iterations` x `num_mini_batches`
                             mini-batch steps, policy net `train_pi_iterations` full-batch steps,
                             gradients averaged across ranks (mpi_avg_grads, mpi_tools.py:30-36)
  algs/ppo/ppo.py:22-40      clipped surrogate loss (clip_ratio=None: IWPG's unclipped -(r A).mean(),
                             algs/iwpg/iwpg.py compute_loss_pi)
  algs/ppo/defaults.py:6-19  networks pi 50-50 relu, v 64-64 tanh, gamma 0.99
The env.step hot path, GAE, running statistics and the fused policy step are CUDA kernels of this
repo.  The update's losses and gradients run as torch autograd (update_kernel='torch', the default and
the reference the tests compare against) or in the fused kernels pdx_ppo_pi_grad / pdx_ppo_v_grad
(update_kernel='cuda'), which fill p.grad directly; Adam, the mini-batches and the schedule stay torch
either way.  Ranks: one process per GPU, NCCL all-reduce of gradients.
"""
import ctypes as C
import math
import time

import torch

from . import lib as _lib
from .rollout import ActorCritic, RolloutCollector, _world
from .vec_env import VecEnv

UPDATE_KERNELS = ('torch', 'cuda')


def check_update_kernel_plan(ac):
    """ValueError unless pdx_ppo_pi_grad / pdx_ppo_v_grad support the networks of `ac`: two hidden layers of <= 64
    units, 4 actions, obs_dim <= 384, float32 parameters."""
    lins = lambda net: [m for m in net if isinstance(m, torch.nn.Linear)]
    pi, v = lins(ac.pi), lins(ac.v)
    obs_dim = pi[0].in_features
    for name, ls, n_out in (('actor', pi, 4), ('critic', v, 1)):
        if len(ls) != 3 or ls[-1].out_features != n_out or not all(1 <= m.out_features <= 64 for m in ls[:2]):
            raise ValueError(f'update_kernel=cuda: the {name} must have two hidden layers of <= 64 units and '
                             f'{n_out} output(s); got {[m.out_features for m in ls]}')
        if any(m.weight.dtype != torch.float32 for m in ls):
            raise ValueError(f'update_kernel=cuda: the {name} must have float32 parameters')
    if not 1 <= obs_dim <= 384:
        raise ValueError(f'update_kernel=cuda: obs_dim must be in [1, 384]; got {obs_dim}')


def _grad_struct(net):
    """PdxMlpGrad over p.grad of the three nn.Linear layers, allocated where missing (the kernel overwrites every
    entry, so no zeroing is needed)."""
    g = _lib.PdxMlpGrad()
    for k, lin in enumerate(m for m in net if isinstance(m, torch.nn.Linear)):
        for p_ in (lin.weight, lin.bias):
            if p_.grad is None:
                p_.grad = torch.empty_like(p_)
        g.weight[k], g.bias[k] = lin.weight.grad.data_ptr(), lin.bias.grad.data_ptr()
    return g


def _prepare(ac, net, n_out, obs, index):
    check_update_kernel_plan(ac)
    if not obs.is_cuda:
        raise ValueError('update_kernel=cuda needs CUDA tensors')
    assert obs.dtype == torch.float32 and obs.is_contiguous() and obs.dim() == 2
    mlp = ac._mlp_struct(net, n_out)
    b = _lib.PdxPpoBatch()
    b.n = obs.shape[0] if index is None else index.shape[0]
    b.obs_dim, b.obs = obs.shape[1], obs.data_ptr()
    if index is not None:
        assert index.dtype == torch.int64 and index.is_contiguous() and index.device == obs.device
        b.index = index.data_ptr()
    L = _lib.load()
    key = (obs.device, obs.shape[1], n_out, tuple(mlp.hidden))
    cache = ac.__dict__.setdefault('_ppo_scratch', {})
    if key not in cache:
        nbytes = int(L.pdx_ppo_scratch_bytes(obs.device.index or 0, obs.shape[1], C.byref(mlp)))
        if nbytes < 0:
            _lib.check(nbytes)
        cache[key] = torch.empty(nbytes, dtype=torch.uint8, device=obs.device)
    scratch = cache[key]
    st = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
    return L, b, mlp, scratch, st


def _vec(t, rows, what):
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape[0] == rows, what
    return t.data_ptr()


def pi_loss_and_grad(ac, obs, act, adv, logp_old, clip_ratio, index=None, grad=True, mu=None, mu_ref=None):
    """PPO's clipped surrogate loss of the actor (algs/ppo/ppo.py:22-40, without the entropy term) in ONE fused CUDA
    kernel (pdx_ppo_pi_grad); clip_ratio None (or inf): the unclipped -(r A).mean() of IWPG / NPG / TRPO.  obs [rows, D] standardised, act [rows, 4], adv / logp_old [rows], float32 CUDA;
    optional int64 `index` [n] selects the rows.  grad=True writes d loss / d weight and bias into p.grad of ac.pi's
    nn.Linear layers (log_std is frozen and gets none).  mu [n, 4]: receives pi(obs).  mu_ref [n, 4]: the Gaussian
    KL mean_i sum_j (mu_ref - mu)^2 / (2 std^2) is computed too.  Returns (loss, kl): 0-d float32 device tensors
    (kl None without mu_ref); nothing is read back to the host."""
    L, b, mlp, scratch, st = _prepare(ac, ac.pi, 4, obs, index)
    rows = obs.shape[0]
    b.act, b.adv, b.logp_old = _vec(act, rows, 'act'), _vec(adv, rows, 'adv'), _vec(logp_old, rows, 'logp_old')
    loss = torch.empty((), dtype=torch.float32, device=obs.device)
    kl = torch.empty((), dtype=torch.float32, device=obs.device) if mu_ref is not None else None
    g = _grad_struct(ac.pi) if grad else None
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    for t in (mu, mu_ref):
        assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == (b.n, 4))
    clip = math.inf if clip_ratio is None else float(clip_ratio)
    _lib.check(L.pdx_ppo_pi_grad(C.byref(b), C.byref(mlp), p(ac.log_std.data), clip,
                                 C.byref(g) if g is not None else None, p(loss), p(mu), p(mu_ref), p(kl),
                                 p(scratch), scratch.numel(), st))
    return loss, kl


def pi_net_params(ac):
    """The actor's nn.Linear tensors in the order of the reference's get_flat_params_from(ac.pi.net): W1, b1, W2, b2,
    W3, b3.  log_std (in ac.pi.parameters(), frozen) is not among them."""
    return [p_ for m in ac.pi if isinstance(m, torch.nn.Linear) for p_ in (m.weight, m.bias)]


def flat_views(flat, params):
    """Views into the flat vector `flat`, one per tensor of `params`, in order and with their shapes."""
    out, k = [], 0
    for p_ in params:
        out.append(flat[k:k + p_.numel()].view_as(p_))
        k += p_.numel()
    assert k == flat.numel(), (k, flat.numel())
    return out


def pi_flat_params(ac):
    return torch.cat([p_.detach().reshape(-1) for p_ in pi_net_params(ac)])


def set_pi_flat_params(ac, flat):
    with torch.no_grad():
        for p_, v in zip(pi_net_params(ac), flat_views(flat, pi_net_params(ac))):
            p_.copy_(v)


def pi_fvp_torch(ac, obs, direction, damping, scale, index=None):
    """The reference's Fvp (algs/npg/npg.py) restated literally: the double backward of the mean per-dimension Normal
    KL of the detached current policy to itself, applied to `direction`, plus damping * direction.  scale 1/4 is that
    KL (its mean runs over the 4 action dimensions too); another scale multiplies it by 4 * scale."""
    params = pi_net_params(ac)
    o = obs if index is None else obs[index]
    mu = ac.pi(o)
    std = torch.exp(ac.log_std).to(mu.dtype)
    q_dist = torch.distributions.Normal(mu, std)
    with torch.no_grad():
        p_dist = torch.distributions.Normal(mu.detach(), std)
    kl = torch.distributions.kl.kl_divergence(p_dist, q_dist).mean() * (scale * mu.shape[-1])
    grads = torch.autograd.grad(kl, params, create_graph=True)
    flat_grad_kl = torch.cat([g.view(-1) for g in grads])
    kl_p = (flat_grad_kl * direction).sum()
    grads = torch.autograd.grad(kl_p, params, retain_graph=False)
    return torch.cat([g.contiguous().view(-1) for g in grads]) + direction * damping


def pi_fvp(ac, obs, direction, damping, scale, index=None, out=None):
    """Fisher-vector product of the actor in ONE fused CUDA kernel (pdx_ppo_pi_fvp):
        scale * (1/n) sum_i J_i^T diag(std^-2) J_i direction + damping * direction,  J_i = d pi(obs_i) / d theta
    = scale x the Hessian of pi_loss_and_grad's kl (sum over the 4 action dimensions) applied to `direction`, plus
    damping; scale = 1/4 is the reference's Fvp (pi_fvp_torch).  direction / out: flat float32 CUDA vectors in the
    order of pi_net_params; the kernel reads and writes them through views, without copies.  Optional int64 `index`
    selects the rows (NPG: every 4th).  Returns `out` (allocated when None); nothing is read back to the host."""
    L, b, mlp, scratch, st = _prepare(ac, ac.pi, 4, obs, index)
    params = pi_net_params(ac)
    assert direction.is_cuda and direction.dtype == torch.float32 and direction.is_contiguous() and direction.dim() == 1
    out = torch.empty_like(direction) if out is None else out
    assert out.dtype == torch.float32 and out.is_contiguous() and out.shape == direction.shape
    d = _lib.PdxMlp()
    d.hidden[0], d.hidden[1], d.n_out = mlp.hidden[0], mlp.hidden[1], 4
    g = _lib.PdxMlpGrad()
    dv, ov = flat_views(direction, params), flat_views(out, params)
    for k in range(3):
        d.weight[k], d.bias[k] = dv[2 * k].data_ptr(), dv[2 * k + 1].data_ptr()
        g.weight[k], g.bias[k] = ov[2 * k].data_ptr(), ov[2 * k + 1].data_ptr()
    _lib.check(L.pdx_ppo_pi_fvp(C.byref(b), C.byref(mlp), C.c_void_p(ac.log_std.data.data_ptr()), C.byref(d),
                                float(scale), float(damping), C.byref(g), C.c_void_p(scratch.data_ptr()),
                                scratch.numel(), st))
    return out


def v_loss_and_grad(ac, obs, target_v, index=None):
    """The value loss mean((v(obs) - target_v)^2) (algs/iwpg/iwpg.py:446-485) in ONE fused CUDA kernel
    (pdx_ppo_v_grad), its gradient written into p.grad of ac.v's nn.Linear layers.  obs [rows, D], target_v [rows]
    float32 CUDA; optional int64 `index` [n] (a mini-batch perm[start:start + mbs], read in place).  Returns the
    loss as a 0-d float32 device tensor."""
    L, b, mlp, scratch, st = _prepare(ac, ac.v, 1, obs, index)
    b.target_v = _vec(target_v, obs.shape[0], 'target_v')
    loss = torch.empty((), dtype=torch.float32, device=obs.device)
    g = _grad_struct(ac.v)
    _lib.check(L.pdx_ppo_v_grad(C.byref(b), C.byref(mlp), C.byref(g), C.c_void_p(loss.data_ptr()),
                                C.c_void_p(scratch.data_ptr()), scratch.numel(), st))
    return loss


class PPO:
    def __init__(self, env_id, num_envs=4096, steps=64, epochs=50, device='cuda', seed=0, dist=None,
                 gamma=0.99, lam=0.95, clip_ratio=0.2, pi_lr=3e-4, vf_lr=1e-3, train_pi_iterations=80,
                 train_v_iterations=5, num_mini_batches=16, entropy_coef=0.0, target_kl=0.01,
                 use_kl_early_stopping=False, use_linear_lr_decay=True, use_exploration_noise_anneal=True,
                 use_standardized_advantages=False, update_kernel='torch', **env_kwargs):
        # update_kernel: 'torch' = autograd; 'cuda' = the fused loss-and-gradient kernels (pdx_ppo_pi_grad /
        # pdx_ppo_v_grad) fill p.grad, everything else in update() stays the same
        if update_kernel not in UPDATE_KERNELS:
            raise ValueError(f'update_kernel must be one of {UPDATE_KERNELS}; got {update_kernel!r}')
        if update_kernel == 'cuda' and torch.device(device).type != 'cuda':
            raise ValueError(f"update_kernel='cuda' needs a CUDA device; got {device!r}")
        self.update_kernel = update_kernel
        rank = dist.get_rank() if _world(dist) > 1 else 0
        self.dist, self.epochs, self.epoch = dist, epochs, 0
        self.env = VecEnv(env_id, num_envs, device=device, seed=seed, env_offset=rank * num_envs,
                          keep_final_obs=True, **env_kwargs)
        torch.manual_seed(seed)                              # same initial weights on every rank (sync_params)
        self.ac = ActorCritic(self.env.obs_dim, device=self.env.device, dist=dist, seed=seed + 10000 * rank)
        if update_kernel == 'cuda':
            check_update_kernel_plan(self.ac)
        # The reference resets the env at the start of every roll_out and demands max_ep_len <=
        # local_steps_per_epoch (iwpg.py:217,353).  With a shorter rollout window that would only ever show
        # the first `steps` steps of an episode, so episodes then continue across rollouts (the collector
        # carries obs[T] and bootstraps the cut with V(obs[T]), iwpg.py:376-378).
        self.collector = RolloutCollector(self.env, self.ac, steps, gamma=gamma, lam=lam, dist=dist,
                                          reset_each_rollout=steps >= self.env.max_episode_steps)
        # clip_ratio None: the unclipped surrogate -(r A).mean() (the reference's IWPG)
        self.clip_ratio, self.entropy_coef, self.target_kl = clip_ratio, entropy_coef, target_kl
        self.train_pi_iterations, self.train_v_iterations = train_pi_iterations, train_v_iterations
        self.num_mini_batches, self.use_kl_early_stopping = num_mini_batches, use_kl_early_stopping
        self.use_exploration_noise_anneal = use_exploration_noise_anneal
        self.use_standardized_advantages = use_standardized_advantages
        self.pi_opt = torch.optim.Adam(self.ac.pi.parameters(), lr=pi_lr)
        self.vf_opt = torch.optim.Adam(self.ac.v.parameters(), lr=vf_lr)
        self.sched = None
        if use_linear_lr_decay:                              # iwpg.py:208-221
            self.sched = torch.optim.lr_scheduler.LambdaLR(self.pi_opt, lambda e: 1 - e / max(1, epochs))
        self.history = []

    # ---------------------------------------------------------------------------------------
    def _avg_grads(self, module):
        P = _world(self.dist)
        if P > 1:
            for p in module.parameters():
                if p.grad is None:                       # the frozen log_std
                    continue
                self.dist.all_reduce(p.grad, op=self.dist.ReduceOp.SUM)
                p.grad /= P

    def _log_prob(self, obs_std, act):
        mu = self.ac.pi(obs_std)
        std = torch.exp(self.ac.log_std)
        logp = (-0.5 * ((act - mu) / std) ** 2 - self.ac.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        return mu, std, logp

    def _loss_pi(self, obs, act, adv, logp_old):            # ppo.py:22-40
        mu, std, logp = self._log_prob(obs, act)
        ratio = torch.exp(logp - logp_old)
        if self.clip_ratio is None:                         # iwpg.py compute_loss_pi
            loss = -(ratio * adv).mean()
        else:
            clip_adv = adv * torch.clamp(ratio, 1 - self.clip_ratio, 1 + self.clip_ratio)
            loss = -torch.min(ratio * adv, clip_adv).mean()
        if self.entropy_coef:
            # ppo.py:32: `loss_pi -= entropy_coef * dist.entropy().mean()` -- the mean over the batch AND the
            # action dimensions of the per-dimension Gaussian entropy
            loss = loss - self.entropy_coef * (0.5 + 0.5 * math.log(2 * math.pi) + self.ac.log_std).mean()
        return loss, mu, std

    def update(self, data):
        T, N = data['rew'].shape
        obs = self.ac.obs_oms(data['obs'].reshape(T * N, -1).float())       # pre_process_data
        act, adv = data['act'].reshape(T * N, -1), data['adv'].reshape(-1)
        target_v, logp_old = data['target_v'].reshape(-1), data['log_p'].reshape(-1)
        if self.use_standardized_advantages:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        loss_v = self.update_v(obs, target_v)
        loss_pi, it, kl = self.update_pi(obs, act, adv, logp_old)
        return {'loss_v': float(loss_v.detach()), 'loss_pi': float(loss_pi.detach()), 'pi_iters': it + 1, 'kl': kl}

    def update_v(self, obs, target_v):
        """Value net: mini-batch steps (iwpg.py:446-485).  Returns the last mini-batch's loss (device tensor)."""
        n = obs.shape[0]
        mbs = n // self.num_mini_batches
        cuda = self.update_kernel == 'cuda'
        if cuda:
            obs, target_v = obs.contiguous(), target_v.contiguous()
        for _ in range(self.train_v_iterations):
            perm = torch.randperm(n, device=obs.device)
            for start in range(0, mbs * self.num_mini_batches, mbs):
                idx = perm[start:start + mbs]
                if cuda:                                 # the kernel overwrites every gradient entry
                    loss_v = v_loss_and_grad(self.ac, obs, target_v, idx)
                else:
                    self.vf_opt.zero_grad(set_to_none=True)
                    loss_v = ((self.ac.v(obs[idx]).squeeze(-1) - target_v[idx]) ** 2).mean()
                    loss_v.backward()
                self._avg_grads(self.ac.v)
                self.vf_opt.step()
        return loss_v

    def _pi_forward(self, obs, act, adv, logp_old, mu_ref=None):
        """(mu, kl) of the current actor, no gradients."""
        if self.update_kernel == 'cuda':
            mu = torch.empty((obs.shape[0], 4), dtype=torch.float32, device=obs.device)
            _, kl = pi_loss_and_grad(self.ac, obs, act, adv, logp_old, self.clip_ratio, grad=False, mu=mu, mu_ref=mu_ref)
            return mu, kl
        with torch.no_grad():
            mu, std, _ = self._log_prob(obs, act)
            if mu_ref is None:
                return mu, None
            # log(std_n / std_old) + (std_old^2 + (mu_old - mu_n)^2) / (2 std_n^2) - 1/2 with std_n == std_old: log_std
            # is frozen during an update
            k = torch.log(std / std) + (std ** 2 + (mu_ref - mu) ** 2) / (2 * std ** 2) - 0.5
            return mu, k.sum(-1).mean()

    def update_pi(self, obs, act, adv, logp_old):
        """Policy net: full-batch steps (iwpg.py:416-444).  Returns (last loss as a device tensor, last iteration, kl)."""
        cuda = self.update_kernel == 'cuda'
        if cuda:
            obs, act, adv, logp_old = obs.contiguous(), act.contiguous(), adv.contiguous(), logp_old.contiguous()
        mu_old = self._pi_forward(obs, act, adv, logp_old)[0] if (self.use_kl_early_stopping or not cuda) else None
        kl, it = 0.0, 0
        for it in range(self.train_pi_iterations):
            if cuda:
                loss_pi, _ = pi_loss_and_grad(self.ac, obs, act, adv, logp_old, self.clip_ratio)
                if self.entropy_coef:                    # a constant: log_std is frozen
                    loss_pi = loss_pi - self.entropy_coef * (0.5 + 0.5 * math.log(2 * math.pi) + self.ac.log_std).mean()
            else:
                self.pi_opt.zero_grad(set_to_none=True)
                loss_pi, mu, std = self._loss_pi(obs, act, adv, logp_old)
                loss_pi.backward()
            self._avg_grads(self.ac.pi)
            self.pi_opt.step()
            if self.use_kl_early_stopping:
                kl_t = self._pi_forward(obs, act, adv, logp_old, mu_ref=mu_old)[1].reshape(1)
                if _world(self.dist) > 1:
                    self.dist.all_reduce(kl_t)
                    kl_t /= _world(self.dist)
                kl = float(kl_t)
                if kl > self.target_kl:
                    break
        return loss_pi, it, kl

    def learn_one_epoch(self):
        t0 = time.perf_counter()
        if self.use_exploration_noise_anneal:                # iwpg.py:272-273
            self.ac.set_log_std(1 - self.epoch / max(1, self.epochs))
        data = self.collector.collect()
        info = self.update(data)
        self.collector.update_running_statistics(data)       # after the update, on the raw data
        if self.sched is not None:
            self.sched.step()
        torch.cuda.synchronize(self.env.device)
        dt = time.perf_counter() - t0
        T, N = data['rew'].shape
        es = data['episode_stats']
        row = dict(epoch=self.epoch, EpRet=es.ret_mean, EpLen=es.len_mean, episodes=es.n,
                   FPS=T * N * _world(self.dist) / dt, **info)
        self.history.append(row)
        self.epoch += 1
        return row

    def learn(self, verbose=False):
        for _ in range(self.epochs):
            row = self.learn_one_epoch()
            if verbose:
                print({k: (round(v, 4) if isinstance(v, float) else v) for k, v in row.items()}, flush=True)
        return self.ac, self.env


def learn(env_id, **kwargs):
    """Counterpart of algs/ppo/ppo.py:50-63 `learn(env_id, **kwargs) -> (ac, env)`."""
    return PPO(env_id, **kwargs).learn()
