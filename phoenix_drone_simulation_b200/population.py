"""A population of PPO agents trained in one process on one GPU (seed sweeps such as the reference's experiment 07).

P members share one env configuration.  Member m owns environments [m N, (m + 1) N) of one VecEnv of P N
environments and has its own networks, Adam state, observation / return normalisers and mini-batch permutations.
The environment and policy-noise draws are keyed by the global environment index, so member m is exactly the single
agent that `VecEnv(num_envs=N, env_offset=m N)`, `ActorCritic(policy_kernel='cuda')` with the same weights and the
same normaliser state would give (see tests/test_gpu_population.py).

Every per-member step of ppo.PPO becomes one launch for all members: the policy step (pdx_policy_step_members),
GAE (pdx_gae_members), the observation moments (pdx_moments_members) and, with update_kernel='cuda', the losses and
gradients (pdx_ppo_pi_grad_members / pdx_ppo_v_grad_members).  update_kernel='torch' computes the same update with
batched matrix products and autograd over the stacked parameters; it is the reference the kernels are tested against.

PopulationNPG / PopulationTRPO do the same for npg.NPG / trpo.TRPO: one surrogate-gradient launch, one Fisher-vector
product launch per conjugate-gradient iteration (pdx_ppo_pi_fvp_members) and one forward launch per line-search
candidate for all members, each member following the single agent's algorithm step for step.
"""
import ctypes as C
import math
import time

import torch

from . import lib as _lib
from .npg import KL_SCALE
from .ppo import UPDATE_KERNELS, check_update_kernel_plan
from .rollout import ActorCritic, _world
from .vec_env import VecEnv


def _lins(net):
    return [m for m in net if isinstance(m, torch.nn.Linear)]


class StackedAdam:
    """torch.optim.Adam's arithmetic over parameters stacked along a leading member dimension [P, ...] in one fused
    kernel launch per tensor (pdx_adam_members), with one step count per member: a member masked out of a step keeps
    its parameters, moments and step count, so it keeps its own bias correction."""

    def __init__(self, params, members, betas=(0.9, 0.999), eps=1e-8):
        self.params, self.betas, self.eps = list(params), betas, eps
        dev = self.params[0].device
        self.steps = torch.zeros(members, dtype=torch.float64, device=dev)
        self.exp_avg = [torch.zeros_like(p) for p in self.params]
        self.exp_avg_sq = [torch.zeros_like(p) for p in self.params]

    @torch.no_grad()
    def step(self, lr, active=None):
        """lr: float; active: optional [P] bool device tensor (None: every member steps)."""
        self.steps += 1.0 if active is None else active.double()
        L, P = _lib.load(), self.steps.shape[0]
        st = C.c_void_p(torch.cuda.current_stream(self.steps.device).cuda_stream)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        for w, m, v in zip(self.params, self.exp_avg, self.exp_avg_sq):
            _lib.check(L.pdx_adam_members(P, w.numel() // P, p(w), p(w.grad), p(m), p(v), p(self.steps), p(active),
                                          float(lr), self.betas[0], self.betas[1], self.eps, st))


class PopulationPPO:
    def __init__(self, env_id, members=4, num_envs_per_member=512, steps=64, epochs=50, device='cuda', seed=0,
                 dist=None, gamma=0.99, lam=0.95, clip_ratio=0.2, pi_lr=3e-4, vf_lr=1e-3, train_pi_iterations=80,
                 train_v_iterations=5, num_mini_batches=16, entropy_coef=0.0, target_kl=0.01,
                 use_kl_early_stopping=False, use_linear_lr_decay=True, use_exploration_noise_anneal=True,
                 use_standardized_advantages=False, update_kernel='torch', **env_kwargs):
        if update_kernel not in UPDATE_KERNELS:
            raise ValueError(f'update_kernel must be one of {UPDATE_KERNELS}; got {update_kernel!r}')
        if _world(dist) > 1:
            raise ValueError(f'PopulationPPO runs on one GPU; got a process group of {_world(dist)} ranks '
                             '(train one population per GPU instead)')
        if int(members) < 1 or int(num_envs_per_member) < 1:
            raise ValueError('members and num_envs_per_member must be >= 1')
        if torch.device(device).type != 'cuda':
            raise ValueError(f'PopulationPPO needs a CUDA device; got {device!r}')
        # the member kernels read the rollout's observations and rewards as float32
        if env_kwargs.get('dtype', torch.float32) != torch.float32:
            raise ValueError(f"PopulationPPO runs float32 environments; got dtype={env_kwargs['dtype']!r}")
        if env_kwargs.get('rng', 'philox') != 'philox':
            raise ValueError(f"PopulationPPO draws on the device (rng='philox'); got rng={env_kwargs['rng']!r}")
        self.P, self.N, self.T = int(members), int(num_envs_per_member), int(steps)
        self.update_kernel, self.epochs, self.epoch, self.seed = update_kernel, epochs, 0, int(seed)
        self.env = VecEnv(env_id, self.P * self.N, device=device, seed=seed, keep_final_obs=True, **env_kwargs)
        self.device, D = self.env.device, self.env.obs_dim
        # member m's initial networks are those PPO(seed=seed + m) builds
        acs = []
        for m in range(self.P):
            torch.manual_seed(self.seed + m)
            acs.append(ActorCritic(D, device=self.device, seed=self.seed, policy_kernel='cuda'))
        if update_kernel == 'cuda':
            check_update_kernel_plan(acs[0])
        stack = lambda ts: torch.stack([t.detach() for t in ts]).contiguous()
        self.pi_params, self.v_params = [], []
        for name, out in (('pi', self.pi_params), ('v', self.v_params)):
            for k in range(3):
                for attr in ('weight', 'bias'):
                    out.append(stack([getattr(_lins(getattr(ac, name))[k], attr) for ac in acs]).requires_grad_(True))
        self.pi_hidden = tuple(self.pi_params[2 * k].shape[1] for k in range(2))
        self.v_hidden = tuple(self.v_params[2 * k].shape[1] for k in range(2))
        self.log_std = stack([ac.log_std for ac in acs])
        oms0, roms0 = acs[0].obs_oms, acs[0].ret_oms
        self.obs_eps, self.ret_eps = oms0.eps, roms0.eps
        self.obs_mean, self.obs_std = stack([oms0.mean] * self.P), stack([oms0.std] * self.P)
        self.obs_count = stack([oms0.count] * self.P)                         # [P, 1]
        self.ret_mean, self.ret_std = stack([roms0.mean] * self.P), stack([roms0.std] * self.P)
        self.ret_count = stack([roms0.count] * self.P)
        self._bm = torch.empty(D, dtype=torch.float32, device=self.device)
        self._bv = torch.empty(D, dtype=torch.float32, device=self.device)
        self._counter = 0                                                    # Philox position of the policy noise
        self.gamma, self.lam = gamma, lam
        self.reset_each_rollout = self.T >= self.env.max_episode_steps        # as PPO / RolloutCollector
        self.clip_ratio, self.entropy_coef, self.target_kl = clip_ratio, entropy_coef, target_kl
        self.train_pi_iterations, self.train_v_iterations = train_pi_iterations, train_v_iterations
        self.num_mini_batches, self.use_kl_early_stopping = num_mini_batches, use_kl_early_stopping
        self.use_exploration_noise_anneal = use_exploration_noise_anneal
        self.use_standardized_advantages = use_standardized_advantages
        self.use_linear_lr_decay = use_linear_lr_decay
        self.pi_lr, self.vf_lr = pi_lr, vf_lr
        self._scratch_bufs = {}
        self.pi_opt = StackedAdam(self.pi_params, self.P)
        self.vf_opt = StackedAdam(self.v_params, self.P)
        self._alloc_rollout()
        self.history = []

    # ---- C structs ------------------------------------------------------------------------------
    def _mlp(self, params, n_out):
        st = _lib.PdxMlp()
        st.hidden[0], st.hidden[1], st.n_out = params[0].shape[-2], params[2].shape[-2], n_out
        for k in range(3):
            st.weight[k], st.bias[k] = params[2 * k].data_ptr(), params[2 * k + 1].data_ptr()
        return st

    def _grad(self, params):
        g = _lib.PdxMlpGrad()
        for k in range(3):
            for j, attr in ((2 * k, 'weight'), (2 * k + 1, 'bias')):
                if params[j].grad is None:
                    params[j].grad = torch.empty_like(params[j])
                getattr(g, attr)[k] = params[j].grad.data_ptr()
        return g

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- policy ---------------------------------------------------------------------------------
    def _alloc_rollout(self):
        T, n, D, dev, dt = self.T, self.P * self.N, self.env.obs_dim, self.device, self.env.dtype
        z = lambda *s, dtype=torch.float32: torch.zeros(s, dtype=dtype, device=dev)
        self.obs, self.act = z(T + 1, n, D, dtype=dt), z(T, n, 4)
        self.rew, self.cost = z(T, n, dtype=dt), z(T, n, dtype=dt)
        self.val, self.logp, self.boot = z(T, n), z(T, n), z(T, n)
        self.term, self.trunc = z(T, n, dtype=torch.uint8), z(T, n, dtype=torch.uint8)
        self.ep_ret, self.ep_len = z(T, n, dtype=dt), z(T, n, dtype=torch.int32)
        self.last_val = z(n)
        self._v_act, self._v_logp = z(n, 4), z(n)                             # discarded outputs of value()
        self._started = False
        L = _lib.load()
        self._pi_mlp, self._v_mlp = self._mlp(self.pi_params, 4), self._mlp(self.v_params, 1)
        self.pack_words = int(L.pdx_policy_pack_words(D, C.byref(self._pi_mlp), C.byref(self._v_mlp)))
        _lib.check(min(self.pack_words, 0))
        self.packed = torch.empty((self.P, self.pack_words), dtype=torch.float32, device=dev)
        outs = [{'obs': self.obs[t + 1], 'reward': self.rew[t], 'cost': self.cost[t], 'terminated': self.term[t],
                 'truncated': self.trunc[t], 'episode_return': self.ep_ret[t], 'episode_length': self.ep_len[t]}
                for t in range(T)]
        # the launch right before each env.step is the policy step, which does not write the env state
        self._env_steps = [self.env.prepare_step(self.act[t], outs[t], state_stable=True) for t in range(T)]

    def refresh_packed_weights(self):
        """pdx_policy_pack image of every member: call after the weights changed."""
        L, st = _lib.load(), self._stream()
        D = self.env.obs_dim
        with torch.no_grad():
            for m in range(self.P):
                pi = self._mlp([p[m] for p in self.pi_params], 4)
                v = self._mlp([p[m] for p in self.v_params], 1)
                _lib.check(L.pdx_policy_pack(D, C.byref(pi), C.byref(v), C.c_void_p(self.packed[m].data_ptr()), st))

    def _policy_step(self, obs, act, val, logp, counter, stream):
        """pdx_policy_step_members on obs [P N, D] (member-major) into act / val / logp."""
        p = lambda t: C.c_void_p(t.data_ptr())
        rc = _lib.load().pdx_policy_step_members(
            self.P, self.N, self.env.obs_dim, p(obs), p(self.obs_mean), p(self.obs_std), self.obs_eps,
            C.byref(self._pi_mlp), C.byref(self._v_mlp), p(self.log_std), p(self.packed), self.pack_words, self.seed,
            counter, self.env.env_offset, p(act), p(val), p(logp), None, stream)
        if rc:
            _lib.check(rc)

    @torch.no_grad()
    def value(self, obs, out):
        """V(obs) of every member's rows of obs [P N, D] into out [P N] (the policy step at counter 0, its action
        draw discarded, as ActorCritic.value)."""
        self._policy_step(obs.contiguous(), self._v_act, out, self._v_logp, 0, self._stream())
        return out

    # ---- rollout ----------------------------------------------------------------------------------
    @torch.no_grad()
    def collect(self):
        """One rollout of T steps of every member: RolloutCollector.collect's loop with the member policy step."""
        env, T = self.env, self.T
        if self.reset_each_rollout or not self._started:
            self.obs[0].copy_(env.reset())
            self._started = True
        else:
            self.obs[0].copy_(self.obs[T])
        env.clear_episode_stats()
        self.boot.zero_()
        self.refresh_packed_weights()
        st = self._stream()
        may_trunc = (not self.reset_each_rollout) or bool(env.cfg.reset_on_nonfinite)
        boot_row = torch.empty_like(self.last_val)
        for t in range(T):
            self._counter += 1
            self._policy_step(self.obs[t], self.act[t], self.val[t], self.logp[t], self._counter, st)
            env.step_prepared(self._env_steps[t], st)
            if may_trunc or t + 1 >= env.max_episode_steps:
                self.boot[t] = self.value(env.final_obs, boot_row) * self.trunc[t].float()
        self.value(self.obs[T], self.last_val)
        done = torch.where(self.trunc > 0, torch.full_like(self.term, 2), self.term)
        adv, target_v, disc_ret = self.gae(done)
        return {'obs': self.obs[:T], 'act': self.act, 'adv': adv, 'target_v': target_v, 'log_p': self.logp,
                'discounted_ret': disc_ret, 'rew': self.rew, 'val': self.val, 'done': done,
                'episode_stats': self.episode_stats()}

    def gae(self, done):
        T, n = self.rew.shape
        adv, tv, dr = (torch.empty((T, n), dtype=torch.float32, device=self.device) for _ in range(3))
        p = lambda t: C.c_void_p(t.data_ptr())
        _lib.check(_lib.load().pdx_gae_members(
            self.P, T, self.N, p(self.rew), p(self.val), p(done), p(self.boot), p(self.last_val), self.gamma, self.lam,
            self.ret_eps, 1, p(self.ret_std), p(adv), p(tv), p(dr), self._stream()))
        return adv, tv, dr

    def episode_stats(self):
        """[P, 8] float64 device tensor per member, VecEnv.episode_stats' layout: n, sum ret, sum ret^2, sum len,
        min ret, max ret, min len, max len (1e300 / -1e300 without a finished episode), reduced from the steps'
        episode_return / episode_length outputs over each member's block of environments."""
        P = self.P
        ln = self.ep_len.view(self.T, P, self.N).transpose(0, 1).reshape(P, -1)
        ret = self.ep_ret.view(self.T, P, self.N).transpose(0, 1).reshape(P, -1).double()
        fin = ln > 0
        lnd = ln.double()
        big = torch.full_like(ret, 1e300)
        return torch.stack([fin.double().sum(1), ret.sum(1), (ret * ret).sum(1), lnd.sum(1),
                            torch.where(fin, ret, big).amin(1), torch.where(fin, ret, -big).amax(1),
                            torch.where(fin, lnd, big).amin(1), torch.where(fin, lnd, -big).amax(1)], dim=1)

    @torch.no_grad()
    def update_running_statistics(self, data):
        """iwpg.py:387-396 per member: OnlineMeanStd.update of the observations and the discounted returns."""
        L, st = _lib.load(), self._stream()
        p = lambda t: C.c_void_p(t.data_ptr())
        for x, mean, std, count in ((data['obs'], self.obs_mean, self.obs_std, self.obs_count),
                                    (data['discounted_ret'].unsqueeze(-1), self.ret_mean, self.ret_std, self.ret_count)):
            T, dim = x.shape[0], x.shape[-1]
            x = x.contiguous().float()
            sums = torch.zeros((self.P, 2 * dim), dtype=torch.float64, device=self.device)
            _lib.check(L.pdx_moments_members(self.P, T, self.N, dim, p(x), None, p(sums), st))
            bm, bv = self._bm[:dim], self._bv[:dim]
            for m in range(self.P):
                _lib.check(L.pdx_oms_update(dim, p(sums[m, :dim]), p(sums[m, dim:]), float(T * self.N), 1, None, p(bm),
                                            p(bv), p(mean[m]), p(std[m]), p(count[m]), 3, st))

    # ---- update ------------------------------------------------------------------------------------
    def _member_major(self, x):
        """[T, P N, ...] -> [P, T N, ...] (member m's rows in the order of its own [T, N] rollout)."""
        T = x.shape[0]
        return x.reshape(T, self.P, self.N, *x.shape[2:]).transpose(0, 1).reshape(self.P, T * self.N, *x.shape[2:]).contiguous()

    @staticmethod
    def _forward(params, x, act):
        h = x
        for k in range(3):
            h = torch.baddbmm(params[2 * k + 1].unsqueeze(1), h, params[2 * k].transpose(1, 2))
            if k < 2:
                h = act(h)
        return h

    def _log_prob(self, obs, act):
        mu = self._forward(self.pi_params, obs, torch.relu)
        ls = self.log_std.unsqueeze(1)
        std = torch.exp(ls)
        logp = (-0.5 * ((act - mu) / std) ** 2 - ls - 0.5 * math.log(2 * math.pi)).sum(-1)
        return mu, std, logp

    def _entropy_term(self):
        return self.entropy_coef * (0.5 + 0.5 * math.log(2 * math.pi) + self.log_std).mean(1)

    def _scratch(self, params, n_out):
        """P x pdx_ppo_scratch_bytes() of device scratch for the actor (n_out 4) or the critic (n_out 1), kept."""
        if n_out not in self._scratch_bufs:
            mlp = self._mlp(params, n_out)
            nbytes = int(_lib.load().pdx_ppo_scratch_bytes(self.device.index or 0, self.env.obs_dim, C.byref(mlp)))
            _lib.check(min(nbytes, 0))
            self._scratch_bufs[n_out] = torch.empty(self.P * nbytes, dtype=torch.uint8, device=self.device)
        return self._scratch_bufs[n_out]

    def _batch(self, obs, index):
        b = _lib.PdxPpoBatch()
        b.n = obs.shape[1] if index is None else index.shape[1]
        b.obs_dim, b.obs = obs.shape[2], obs.data_ptr()
        b.index = index.data_ptr() if index is not None else None
        return b

    def pi_loss_and_grad(self, obs, act, adv, logp_old, grad=True, mu=None, mu_ref=None, active=None):
        """pdx_ppo_pi_grad_members: loss [P] (and kl [P] with mu_ref) of every member; grad=True writes the gradients
        into .grad of the stacked actor parameters.  obs [P, n, D], act [P, n, 4], adv / logp_old [P, n]."""
        b = self._batch(obs, None)
        b.act, b.adv, b.logp_old = act.data_ptr(), adv.data_ptr(), logp_old.data_ptr()
        loss = torch.empty(self.P, dtype=torch.float32, device=self.device)
        kl = torch.empty(self.P, dtype=torch.float32, device=self.device) if mu_ref is not None else None
        g = self._grad(self.pi_params) if grad else None
        scratch = self._scratch(self.pi_params, 4)
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        clip = math.inf if self.clip_ratio is None else float(self.clip_ratio)
        _lib.check(_lib.load().pdx_ppo_pi_grad_members(
            self.P, C.byref(b), obs.shape[1], p(active), C.byref(self._mlp(self.pi_params, 4)), p(self.log_std), clip,
            C.byref(g) if g is not None else None, p(loss), p(mu), p(mu_ref), p(kl), p(scratch), scratch.numel(),
            self._stream()))
        return loss, kl

    def v_loss_and_grad(self, obs, target_v, index):
        """pdx_ppo_v_grad_members: loss [P] over the rows index [P, mbs] of every member, gradients into .grad."""
        b = self._batch(obs, index)
        b.target_v = target_v.data_ptr()
        loss = torch.empty(self.P, dtype=torch.float32, device=self.device)
        scratch = self._scratch(self.v_params, 1)
        _lib.check(_lib.load().pdx_ppo_v_grad_members(
            self.P, C.byref(b), obs.shape[1], None, C.byref(self._mlp(self.v_params, 1)),
            C.byref(self._grad(self.v_params)), C.c_void_p(loss.data_ptr()), C.c_void_p(scratch.data_ptr()),
            scratch.numel(), self._stream()))
        return loss

    def update(self, data):
        obs = self._member_major(data['obs'].float())
        obs = (obs - self.obs_mean.unsqueeze(1)) / (self.obs_std.unsqueeze(1) + self.obs_eps)
        act, adv = self._member_major(data['act']), self._member_major(data['adv'])
        target_v, logp_old = self._member_major(data['target_v']), self._member_major(data['log_p'])
        if self.use_standardized_advantages:
            adv = (adv - adv.mean(1, keepdim=True)) / (adv.std(1, keepdim=True) + 1e-8)
        loss_v = self.update_v(obs, target_v)
        loss_pi, iters, kl = self.update_pi(obs, act, adv, logp_old)
        return {'loss_v': loss_v.tolist(), 'loss_pi': loss_pi.tolist(), 'pi_iters': iters, 'kl': kl}

    def update_v(self, obs, target_v):
        """Value nets: train_v_iterations x num_mini_batches steps, each member with its own permutations."""
        P, n = obs.shape[:2]
        mbs = n // self.num_mini_batches
        rows = torch.arange(P, device=obs.device).unsqueeze(1)
        for _ in range(self.train_v_iterations):
            perm = torch.stack([torch.randperm(n, device=obs.device) for _ in range(P)])
            for start in range(0, mbs * self.num_mini_batches, mbs):
                idx = perm[:, start:start + mbs].contiguous()
                if self.update_kernel == 'cuda':
                    loss_v = self.v_loss_and_grad(obs, target_v, idx)
                else:
                    for p_ in self.v_params:
                        p_.grad = None
                    v = self._forward(self.v_params, obs[rows, idx], torch.tanh).squeeze(-1)
                    loss_v = ((v - target_v[rows, idx]) ** 2).mean(1)
                    loss_v.sum().backward()
                self.vf_opt.step(self.vf_lr)
        return loss_v.detach()

    def _pi_forward(self, obs, act, adv, logp_old, mu_ref=None, active=None):
        """(mu, kl) of every member's actor, no gradients."""
        if self.update_kernel == 'cuda':
            mu = torch.empty((self.P, obs.shape[1], 4), dtype=torch.float32, device=obs.device)
            _, kl = self.pi_loss_and_grad(obs, act, adv, logp_old, grad=False, mu=mu, mu_ref=mu_ref, active=active)
            return mu, kl
        with torch.no_grad():
            mu, std, _ = self._log_prob(obs, act)
            if mu_ref is None:
                return mu, None
            k = torch.log(std / std) + (std ** 2 + (mu_ref - mu) ** 2) / (2 * std ** 2) - 0.5
            return mu, k.sum(-1).mean(1)

    def update_pi(self, obs, act, adv, logp_old):
        """Policy nets: full-batch steps; with KL early stopping each member stops at its own iteration and a stopped
        member's actor and Adam state do not move.  Returns (loss [P] of each member's last step, iterations [P],
        kl [P])."""
        P, cuda = self.P, self.update_kernel == 'cuda'
        lr = self.pi_lr * (1 - self.epoch / max(1, self.epochs)) if self.use_linear_lr_decay else self.pi_lr
        mu_old = self._pi_forward(obs, act, adv, logp_old)[0] if self.use_kl_early_stopping else None
        active = torch.ones(P, dtype=torch.bool, device=obs.device) if self.use_kl_early_stopping else None
        last_loss = torch.zeros(P, dtype=torch.float32, device=obs.device)
        iters, kl_out = [self.train_pi_iterations] * P, [0.0] * P
        running = list(range(P))
        for it in range(self.train_pi_iterations):
            if cuda:
                loss_pi, _ = self.pi_loss_and_grad(obs, act, adv, logp_old, active=active)
            else:
                for p_ in self.pi_params:
                    p_.grad = None
                mu, std, logp = self._log_prob(obs, act)
                ratio = torch.exp(logp - logp_old)
                if self.clip_ratio is None:
                    loss_pi = -(ratio * adv).mean(1)
                else:
                    clip_adv = adv * torch.clamp(ratio, 1 - self.clip_ratio, 1 + self.clip_ratio)
                    loss_pi = -torch.min(ratio * adv, clip_adv).mean(1)
                loss_pi.sum().backward()
            if self.entropy_coef:                        # a constant: log_std is frozen
                loss_pi = loss_pi - self._entropy_term()
            loss_pi = loss_pi.detach()
            last_loss = loss_pi if active is None else torch.where(active, loss_pi, last_loss)
            self.pi_opt.step(lr, active)
            if self.use_kl_early_stopping:
                kl = self._pi_forward(obs, act, adv, logp_old, mu_ref=mu_old, active=active)[1].tolist()
                for m in list(running):
                    kl_out[m] = kl[m]
                    if kl[m] > self.target_kl:
                        iters[m] = it + 1
                        running.remove(m)
                if not running:
                    break
                active = torch.zeros(P, dtype=torch.bool)
                active[running] = True
                active = active.to(obs.device)
        return last_loss, iters, kl_out

    # ---- training loop -------------------------------------------------------------------------------
    def learn_one_epoch(self):
        t0 = time.perf_counter()
        if self.use_exploration_noise_anneal:                # iwpg.py:272-273, core.py:268-276
            self.log_std.fill_(math.log(0.499 * (1 - self.epoch / max(1, self.epochs)) + 0.01))
        data = self.collect()
        info = self.update(data)
        self.update_running_statistics(data)                 # after the update, on the raw data
        torch.cuda.synchronize(self.device)
        dt = time.perf_counter() - t0
        es = data['episode_stats'].cpu().tolist()
        ret = [s[1] / s[0] if s[0] else float('nan') for s in es]
        ln = [s[3] / s[0] if s[0] else float('nan') for s in es]
        row = dict(epoch=self.epoch, EpRet=ret, EpLen=ln, episodes=[int(s[0]) for s in es],
                   FPS=self.T * self.N * self.P / dt, **info)
        self.history.append(row)
        self.epoch += 1
        return row

    def learn(self, verbose=False):
        for _ in range(self.epochs):
            row = self.learn_one_epoch()
            if verbose:
                for m in range(self.P):
                    print({'epoch': row['epoch'], 'member': m, 'seed': self.seed + m,
                           **{k: round(row[k][m], 4) if isinstance(row[k][m], float) else row[k][m]
                              for k in ('EpRet', 'EpLen', 'loss_pi', 'loss_v', 'pi_iters', 'kl')}}, flush=True)
        return self

    @torch.no_grad()
    def member(self, m):
        """A standalone ActorCritic (policy_kernel='cuda') with member m's weights, log_std and normalisers: the single
        agent member m is, for policy_io.export_policy_json and policy_io.evaluate_many."""
        with torch.random.fork_rng(devices=[]):       # the weights are overwritten: leave the global RNG alone
            ac = ActorCritic(self.env.obs_dim, device=self.device, seed=self.seed, policy_kernel='cuda')
        for net, params in ((ac.pi, self.pi_params), (ac.v, self.v_params)):
            for k, lin in enumerate(_lins(net)):
                lin.weight.copy_(params[2 * k][m]), lin.bias.copy_(params[2 * k + 1][m])
        ac.pi.log_std.copy_(self.log_std[m])
        for oms, mean, std, count in ((ac.obs_oms, self.obs_mean, self.obs_std, self.obs_count),
                                      (ac.ret_oms, self.ret_mean, self.ret_std, self.ret_count)):
            oms.mean.copy_(mean[m]), oms.std.copy_(std[m]), oms.count.copy_(count[m])
        ac._counter, ac.env_offset = self._counter, self.env.env_offset + m * self.N
        return ac


def conjugate_gradients_members(Avp, b, nsteps, residual_tol=1e-10, eps=1e-6):
    """npg.conjugate_gradients for P independent systems at once: b [P, F], Avp(p, active) -> A_m p_m for every member
    m where active[m] ([P] bool device tensor; rows of inactive members may be left unwritten).  Member m takes exactly
    the single loop's steps (the dot products are row sums, so it agrees to rounding): a member whose residual drops
    below residual_tol keeps that iteration's x and r and drops out, where the single loop breaks, and is inactive in
    the later products.  One host read-back per iteration: whether any member still runs."""
    x = torch.zeros_like(b)
    r = b.clone()
    p = r.clone()
    rdotr = (r * r).sum(1)
    running = torch.ones(b.shape[0], dtype=torch.bool, device=b.device)
    for _ in range(nsteps):
        z = Avp(p, running)
        alpha = (rdotr / ((p * z).sum(1) + eps)).unsqueeze(1)
        live = running.unsqueeze(1)
        x = torch.where(live, x + alpha * p, x)
        r = torch.where(live, r - alpha * z, r)
        new_rdotr = (r * r).sum(1)
        running = running & ~(torch.sqrt(new_rdotr) < residual_tol)
        if not bool(running.any()):
            break
        mu = (new_rdotr / (rdotr + eps)).unsqueeze(1)
        p = torch.where(running.unsqueeze(1), r + mu * p, p)
        rdotr = torch.where(running, new_rdotr, rdotr)
    return x


def line_search_members(evaluate, step, theta_old, target_kl, total_steps=15, decay=0.8):
    """trpo.line_search for P members at once.  step / theta_old [P, F]; evaluate(theta [P, F], active [P] bool device
    tensor) -> (loss improvement [P], kl [P]) as host sequences, read for the active members only.  Candidate j moves
    every member still searching to theta_old + decay^j step; each member accepts the first candidate whose improvement
    is finite and >= 0 and whose kl is <= 1.5 target_kl.  Returns (step to add to theta_old [P, F], accept_step [P]):
    accept_step j + 1 for candidate j, 0 (and a zero step) for a member that passes none.  The fraction is the single
    search's Python float, rounded to float32 as its `frac * step` does."""
    P = step.shape[0]
    fracs, accept = [0.0] * P, [0] * P
    searching = list(range(P))
    frac = 1.0
    for j in range(total_steps):
        active = torch.zeros(P, dtype=torch.bool)
        active[searching] = True
        improve, kl = evaluate(theta_old + frac * step, active.to(step.device))
        for m in list(searching):
            if math.isfinite(improve[m]) and improve[m] >= 0 and kl[m] <= 1.5 * target_kl:
                fracs[m], accept[m] = frac, j + 1
                searching.remove(m)
        if not searching:
            break
        frac *= decay
    f = torch.tensor(fracs, dtype=step.dtype, device=step.device).unsqueeze(1)
    return f * step, accept


class PopulationNPG(PopulationPPO):
    """npg.NPG for a population: PopulationPPO's rollout, value phase and running statistics, and per member exactly
    npg.NPG.update_pi's conjugate-gradient policy step (surrogate gradient g on the full batch, x = CG(F, -g) with the
    Fisher-vector product on every 4th member-local row, step = sqrt(2 target_kl / x^T F x) x).  The actor has no
    optimiser and no learning-rate schedule.  update_kernel='cuda': the gradient is one pdx_ppo_pi_grad_members launch
    and every Fisher-vector product one pdx_ppo_pi_fvp_members launch on the flat [P, F] CG vectors; 'torch': autograd,
    the product being the reference's double backward over the stacked parameters."""

    def __init__(self, env_id, cg_iters=10, cg_damping=0.1, target_kl=0.01, **kwargs):
        super().__init__(env_id, target_kl=target_kl, **kwargs)
        self.clip_ratio = None                               # the unclipped surrogate
        self.cg_iters, self.cg_damping = cg_iters, cg_damping
        self.pi_opt = None                                   # npg.py: no pi optimiser step
        self.step_info = {}

    def update(self, data):
        info = super().update(data)
        info.update(self.step_info)
        return info

    # ---- flat [P, F] parameter vectors, per member in the order of ppo.pi_net_params ----------------------------------
    def _flat_views(self, flat):
        out, k = [], 0
        for p_ in self.pi_params:
            n = p_[0].numel()
            out.append(flat[:, k:k + n].view(p_.shape))
            k += n
        assert k == flat.shape[1], (k, flat.shape)
        return out

    def _flat_params(self):
        return torch.cat([p_.detach().reshape(self.P, -1) for p_ in self.pi_params], 1)

    @torch.no_grad()
    def _set_flat_params(self, flat):
        for p_, v in zip(self.pi_params, self._flat_views(flat)):
            p_.copy_(v)

    # ---- the pieces of the policy step ----------------------------------------------------------------------------------
    def _surrogate_grad(self, obs, act, adv, logp_old):
        """(loss [P], flat gradient [P, F]) of -(r A).mean() on every member's full batch."""
        if self.update_kernel == 'cuda':
            loss, _ = self.pi_loss_and_grad(obs, act, adv, logp_old)
        else:
            for p_ in self.pi_params:
                p_.grad = None
            loss = self._surrogate(obs, act, adv, logp_old)
            loss.sum().backward()
        return loss.detach(), torch.cat([p_.grad.reshape(self.P, -1) for p_ in self.pi_params], 1)

    def _surrogate(self, obs, act, adv, logp_old):
        _, _, logp = self._log_prob(obs, act)
        loss = -(torch.exp(logp - logp_old) * adv).mean(1)
        if self.entropy_coef:
            loss = loss - self._entropy_term()
        return loss

    def _fvp(self, obs, idx, v, active=None):
        """F_m v_m + cg_damping v_m of every member (npg.py Fvp with npg.KL_SCALE), v [P, F]; with update_kernel='cuda'
        the rows of members inactive in `active` are not written."""
        if self.update_kernel == 'cuda':
            out = torch.empty_like(v)
            b = self._batch(obs, idx)
            d, g = _lib.PdxMlp(), _lib.PdxMlpGrad()
            d.hidden[0], d.hidden[1], d.n_out = self.pi_hidden[0], self.pi_hidden[1], 4
            for k, (dv, ov) in enumerate(zip(self._flat_views(v), self._flat_views(out))):
                getattr(d, ('weight', 'bias')[k % 2])[k // 2] = dv.data_ptr()
                getattr(g, ('weight', 'bias')[k % 2])[k // 2] = ov.data_ptr()
            scratch = self._scratch(self.pi_params, 4)
            p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            _lib.check(_lib.load().pdx_ppo_pi_fvp_members(
                self.P, C.byref(b), obs.shape[1], p(active), C.byref(self._mlp(self.pi_params, 4)), p(self.log_std),
                C.byref(d), KL_SCALE, float(self.cg_damping), C.byref(g), v.shape[1], p(scratch), scratch.numel(),
                self._stream()))
            return out
        o = obs[torch.arange(self.P, device=obs.device).unsqueeze(1), idx]
        mu = self._forward(self.pi_params, o, torch.relu)
        std = torch.exp(self.log_std).unsqueeze(1).to(mu.dtype)
        q_dist = torch.distributions.Normal(mu, std)
        with torch.no_grad():
            p_dist = torch.distributions.Normal(mu.detach(), std)
        # the per-member KL means summed: the Hessian is block-diagonal over the members
        kl = (torch.distributions.kl.kl_divergence(p_dist, q_dist).mean((1, 2)) * (KL_SCALE * mu.shape[-1])).sum()
        grads = torch.autograd.grad(kl, self.pi_params, create_graph=True)
        flat_grad_kl = torch.cat([g.reshape(self.P, -1) for g in grads], 1)
        grads = torch.autograd.grad((flat_grad_kl * v).sum(), self.pi_params)
        return torch.cat([g.contiguous().reshape(self.P, -1) for g in grads], 1) + v * self.cg_damping

    def _loss_kl(self, obs, act, adv, logp_old, mu_old, active=None):
        """Forward only: (surrogate loss [P], reference-normalised KL to mu_old [P]) as device tensors; with
        update_kernel='cuda' the entries of members inactive in `active` are not written."""
        if self.update_kernel == 'cuda':
            mu = torch.empty_like(mu_old)
            loss, kl = self.pi_loss_and_grad(obs, act, adv, logp_old, grad=False, mu=mu, mu_ref=mu_old, active=active)
            return loss, kl * KL_SCALE
        with torch.no_grad():
            return self._surrogate(obs, act, adv, logp_old), self._pi_forward(obs, act, adv, logp_old, mu_ref=mu_old)[1] * KL_SCALE

    def search_step_size(self, step, theta_old, evaluate):
        """NPG takes every member's whole natural-gradient step.  Returns (step to add [P, F], accept_step [P])."""
        return step, [1] * self.P

    def update_pi(self, obs, act, adv, logp_old):
        """npg.py update_policy_net per member.  Returns (loss after the step [P], zeros, kl after the step [P])."""
        P, n = obs.shape[:2]
        fvp_idx = torch.arange(0, n, 4, device=obs.device).expand(P, -1).contiguous()
        mu_old = self._pi_forward(obs, act, adv, logp_old)[0]
        theta_old = self._flat_params()
        loss_before, g = self._surrogate_grad(obs, act, adv, logp_old)
        x = conjugate_gradients_members(lambda v, active: self._fvp(obs, fvp_idx, v, active), -g, self.cg_iters)
        xHx = (x * self._fvp(obs, fvp_idx, x)).sum(1)
        step = torch.sqrt(2 * self.target_kl / (xHx + 1e-8)).unsqueeze(1) * x

        def evaluate(theta, active):
            """(loss improvement [P], kl [P]) of every member's actor at theta, as host lists."""
            self._set_flat_params(theta)
            loss, kl = self._loss_kl(obs, act, adv, logp_old, mu_old, active)
            t = torch.stack([loss_before - loss, kl]).tolist()
            return t[0], t[1]

        final_step, accept = self.search_step_size(step, theta_old, evaluate)
        self._set_flat_params(theta_old + final_step)
        loss, kl = self._loss_kl(obs, act, adv, logp_old, mu_old)
        self.step_info = {'accept_step': accept, 'xHx': xHx.tolist()}
        return loss, [0] * P, kl.tolist()


class PopulationTRPO(PopulationNPG):
    """trpo.TRPO for a population: each member's NPG step under trpo.line_search, batched (line_search_members): one
    forward-only pdx_ppo_pi_grad_members launch per candidate for the members still searching."""

    def search_step_size(self, step, theta_old, evaluate):
        return line_search_members(evaluate, step, theta_old, self.target_kl)


def learn(env_id, **kwargs):
    """`ppo.learn` for a population: returns the trained PopulationPPO."""
    return PopulationPPO(env_id, **kwargs).learn()
