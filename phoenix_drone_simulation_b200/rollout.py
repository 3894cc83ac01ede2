"""Device-side PPO rollout collection for the batched engine.

What each piece restates (reference paths relative to phoenix_drone_simulation/):
  ActorCritic        algs/core.py:313-411  (pi 50-50 relu Gaussian, v 64-64 tanh, ppo/defaults.py:6-19;
                     obs standardisation online_mean_std.py:32-48; std annealing core.py:268-276)
  RolloutCollector   algs/iwpg/iwpg.py:350-385 (roll_out) + algs/core.py:481-557 (Buffer) for N
                     lock-step environments: observations never leave device memory, every field
                     is stored time-major in [T, N, .] tensors by the step kernel itself.
  compute_gae        algs/core.py:458-479,497-534 (finish_path) -> CUDA kernel pdx_gae
  OnlineMeanStd      utils/online_mean_std.py:50-95 incl. its non-textbook variance update;
                     the cross-rank averages (mpi_tools.py:199-214) become NCCL all-reduces
  EpisodeStats /     utils/loggers.py:519-524 + mpi_tools.py:217-240 (mean/std/min/max of
  allreduce_episode_stats   EpRet / EpLen across ranks) from the block-reduced sums of the step kernel

Cross-GPU traffic: two small all-reduces per rollout for the episode statistics and two per
`OnlineMeanStd.update` -- nothing on the env.step itself (SURVEY.md 8e).
"""
import ctypes as C
import math

import torch

from . import lib as _lib


def _world(dist):
    return dist.get_world_size() if dist is not None and dist.is_initialized() else 1


# ---------------------------------------------------------------------------------------------
#  episode statistics
# ---------------------------------------------------------------------------------------------
def allreduce_episode_stats(stats, dist):
    """In-place cross-rank combination of the 8-word statistics vector of VecEnv
    [n, sum ret, sum ret^2, sum len, min ret, max ret, min len, max len] (float64): ONE all-gather
    (NCCL) followed by one tiny combine kernel (pdx_stats_combine) on CUDA tensors; on CPU tensors
    (gloo, host-logic tests) the same combination with torch ops."""
    P = _world(dist)
    if P == 1:
        return stats
    flat = torch.empty(P * 8, dtype=torch.float64, device=stats.device)
    dist.all_gather_into_tensor(flat, stats)
    gathered = flat.view(P, 8)
    if stats.is_cuda:
        st = C.c_void_p(torch.cuda.current_stream(stats.device).cuda_stream)
        _lib.check(_lib.load().pdx_stats_combine(P, C.c_void_p(gathered.data_ptr()), C.c_void_p(stats.data_ptr()), st))
    else:
        stats[:4] = gathered[:, :4].sum(0)
        stats[4], stats[6] = gathered[:, 4].min(), gathered[:, 6].min()
        stats[5], stats[7] = gathered[:, 5].max(), gathered[:, 7].max()
    return stats


def gather_episode_stats_async(stats, dist):
    """Asynchronous form of `allreduce_episode_stats`: starts ONE all-gather of the 8-word vector on the
    process group's own stream and returns a function that, when called later, makes the current
    stream wait for it, combines the ranks (pdx_stats_combine) and returns the combined vector.
    The caller keeps launching env.step kernels in between: the collective overlaps them."""
    P = _world(dist)
    if P == 1:
        return lambda: stats
    flat = torch.empty(P * 8, dtype=torch.float64, device=stats.device)
    work = dist.all_gather_into_tensor(flat, stats, async_op=True)

    def finish():
        work.wait()                                      # stream-level wait, the host does not block
        gathered = flat.view(P, 8)
        if stats.is_cuda:
            st = C.c_void_p(torch.cuda.current_stream(stats.device).cuda_stream)
            _lib.check(_lib.load().pdx_stats_combine(P, C.c_void_p(gathered.data_ptr()), C.c_void_p(stats.data_ptr()), st))
        else:
            stats[:4] = gathered[:, :4].sum(0)
            stats[4], stats[6] = gathered[:, 4].min(), gathered[:, 6].min()
            stats[5], stats[7] = gathered[:, 5].max(), gathered[:, 7].max()
        return stats
    return finish


class EpisodeStats:
    """mean / std / min / max of EpRet and mean of EpLen like EpochLogger.get_stats."""

    def __init__(self, stats):
        self._stats = stats                       # device tensor: read back (one sync) when a value is first asked for

    def __getattr__(self, name):
        if name.startswith('_'):
            raise AttributeError(name)
        self._materialise()
        try:
            return self.__dict__[name]
        except KeyError:
            raise AttributeError(name) from None

    def _materialise(self):
        s = [float(v) for v in self._stats.detach().cpu().tolist()]
        self.n = int(s[0])
        if self.n:
            self.ret_mean = s[1] / s[0]
            self.ret_std = math.sqrt(max(s[2] / s[0] - self.ret_mean ** 2, 0.0))   # mpi_tools.py:233
            self.ret_min, self.ret_max = s[4], s[5]
            self.len_mean, self.len_min, self.len_max = s[3] / s[0], s[6], s[7]
        else:
            self.ret_mean = self.ret_std = self.ret_min = self.ret_max = float('nan')
            self.len_mean = self.len_min = self.len_max = float('nan')

    def as_dict(self):
        return {'EpRet/Mean': self.ret_mean, 'EpRet/Std': self.ret_std, 'EpRet/Min': self.ret_min,
                'EpRet/Max': self.ret_max, 'EpLen/Mean': self.len_mean, 'Episodes': self.n}


# ---------------------------------------------------------------------------------------------
#  running mean / std
# ---------------------------------------------------------------------------------------------
def column_moments(x, shift=None):
    """sum_r x[r, :] and sum_r (x[r, :] - shift)^2 in float64 (CUDA kernel pdx_moments)."""
    if not x.is_cuda:
        raise _lib.PhoenixB200Error('column_moments needs CUDA tensors: there is no CPU fallback')
    x = x.reshape(-1, x.shape[-1]).contiguous().float()
    rows, dim = x.shape
    out = torch.zeros(2 * dim, dtype=torch.float64, device=x.device)
    sp = None
    if shift is not None:
        shift = shift.to(device=x.device, dtype=torch.float64).contiguous()
        sp = C.c_void_p(shift.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(_lib.load().pdx_moments(rows, dim, C.c_void_p(x.data_ptr()), sp, C.c_void_p(out.data_ptr()), st))
    return out[:dim], out[dim:]


class OnlineMeanStd(torch.nn.Module):
    """Running mean/std with the reference's update rule (online_mean_std.py:70-95):
    n_B = rows * P; the batch mean is the plain average of the per-rank means; the batch second
    moment is taken about the NEW mean and delta^2 n_A n_B / n_AB is added on top.

    Like the reference's (online_mean_std.py:6-16) this is an nn.Module whose mean / std / count are
    frozen Parameters, so `ActorCritic.state_dict()` carries the normaliser under the reference's key
    names (`obs_oms.mean`, ...).  Updates are in place: prepared launches hold the tensors' addresses."""

    def __init__(self, dim, device, epsilon=1e-5, dist=None, moments_fn=column_moments):
        super().__init__()
        P = lambda t: torch.nn.Parameter(t, requires_grad=False)
        self.mean = P(torch.zeros(dim, dtype=torch.float32, device=device))
        self.std = P(torch.ones(dim, dtype=torch.float32, device=device))
        self.count = P(torch.zeros(1, dtype=torch.float32, device=device))
        self.eps, self.bound, self.dist = epsilon, 10.0, dist
        self._moments = moments_fn

    def forward(self, x, subtract_mean=True, clip=False):
        y = (x - self.mean) / (self.std + self.eps) if subtract_mean else x / (self.std + self.eps)
        return torch.clamp(y, -self.bound, self.bound) if clip else y

    def _avg(self, t):                                   # mpi_tools.mpi_avg_torch_tensor
        P = _world(self.dist)
        if P > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
            t /= P
        return t

    @torch.no_grad()
    def update(self, x):
        x = x.reshape(-1, self.mean.shape[0])
        # ONE pass over the batch: sum x and sum x^2 in float64; the second moment about the new mean
        # follows as sum x^2 - 2 m sum x + rows m^2 (same value as the reference's second pass)
        s1, s2 = self._moments(x, None)
        self.update_from_sums(s1, s2, x.shape[0])

    @torch.no_grad()
    def update_from_sums(self, s1, s2, rows, shift=None):
        """The same update from column sums computed elsewhere (the fused collector kernel accumulates them while
        it rolls out): s1 = sum (x - shift), s2 = sum (x - shift)^2 over `rows` rows, float64.  On CUDA tensors
        the algebra runs in one small kernel (pdx_oms_update) per phase -- one launch for a single rank, three
        with the two rank averages of the reference in between -- instead of ~25 element-wise torch launches."""
        P = _world(self.dist)
        if s1.is_cuda:
            dim = self.mean.shape[0]
            if getattr(self, '_bm', None) is None:
                self._bm = torch.empty(dim, dtype=torch.float32, device=self.mean.device)
                self._bv = torch.empty(dim, dtype=torch.float32, device=self.mean.device)
            p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
            s1, s2 = s1.contiguous(), s2.contiguous()
            sh = shift.float().contiguous() if shift is not None else None
            st = C.c_void_p(torch.cuda.current_stream(s1.device).cuda_stream)
            call = lambda phase: _lib.check(_lib.load().pdx_oms_update(
                dim, p(s1), p(s2), float(rows), P, p(sh), p(self._bm), p(self._bv), p(self.mean.data), p(self.std.data),
                p(self.count.data), phase, st))
            if P == 1:
                call(3)
            else:
                call(0); self._avg(self._bm); call(1); self._avg(self._bv); call(2)
            return
        if shift is not None:
            c = shift.double()
            s2 = s2 + 2.0 * c * s1 + rows * c * c
            s1 = s1 + rows * c
        n_B = float(rows * P)
        n_A = self.count.clone()
        n_AB = self.count + n_B
        batch_mean = self._avg((s1 / rows).float())
        delta = batch_mean - self.mean
        mean_new = self.mean + delta * n_B / n_AB
        m = mean_new.double()
        batch_var = self._avg(((s2 - 2.0 * m * s1 + rows * m * m) / rows).clamp_min(0.0).float())
        M2 = n_A * self.std ** 2 + n_B * batch_var + delta ** 2 * (n_A * n_B / n_AB)
        # in place: prepared launches of the policy kernels hold these tensors
        self.mean.copy_(mean_new)
        self.count.copy_(n_AB)
        self.std.copy_(torch.sqrt(M2 / n_AB))


# ---------------------------------------------------------------------------------------------
#  GAE
# ---------------------------------------------------------------------------------------------
def compute_gae(rew, val, done, boot_val, last_val, gamma=0.99, lam=0.95, ret_std=None, eps=1e-5):
    """Buffer.finish_path for a [T, N] lock-step rollout (CUDA kernel pdx_gae).
    done: uint8, 1 = terminated (v=0), 2 = time limit (bootstrap with boot_val[t]).  `ret_std`:
    running std of the discounted returns -> reward scaling r / (std + eps) clipped to +-10; a
    float, or a one-element float32 CUDA tensor that the kernel reads on the device (no host sync).
    Returns (adv, target_v, discounted_ret), float32 [T, N]."""
    if not rew.is_cuda:
        raise _lib.PhoenixB200Error('compute_gae needs CUDA tensors: there is no CPU fallback')
    T, n = rew.shape
    f = lambda t: t.contiguous().float()
    rew, val, boot_val, last_val = f(rew), f(val), f(boot_val), f(last_val)
    done = done.contiguous().to(torch.uint8)
    adv, tv, dr = torch.empty_like(rew), torch.empty_like(rew), torch.empty_like(rew)
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream(rew.device).cuda_stream)
    std_dev = None
    if torch.is_tensor(ret_std):
        assert ret_std.is_cuda and ret_std.dtype == torch.float32 and ret_std.numel() == 1
        std_dev, scale = p(ret_std), eps
    else:
        scale = float(ret_std) + eps if ret_std is not None else 1.0
    _lib.check(_lib.load().pdx_gae(T, n, p(rew), p(val), p(done), p(boot_val), p(last_val), gamma, lam,
                                   scale, 1 if ret_std is not None else 0, std_dev, p(adv), p(tv), p(dr), st))
    return adv, tv, dr


# ---------------------------------------------------------------------------------------------
#  actor-critic (the reference's PPO networks)
# ---------------------------------------------------------------------------------------------
def _mlp(sizes, act):
    layers = []
    for j in range(len(sizes) - 1):
        lin = torch.nn.Linear(sizes[j], sizes[j + 1])
        torch.nn.init.kaiming_uniform_(lin.weight, a=math.sqrt(5))          # core.py:34-35
        layers += [lin, act() if j < len(sizes) - 2 else torch.nn.Identity()]
    return torch.nn.Sequential(*layers)


class _Net(torch.nn.Module):
    """MLP held under `.net` like the reference's MLPGaussianActor / MLPCritic (core.py:227-310), so
    that state_dict keys read `pi.net.0.weight`, `v.net.4.bias`, ... as in a reference checkpoint."""

    def __init__(self, sizes, act):
        super().__init__()
        self.net = _mlp(sizes, act)

    def forward(self, obs):
        return self.net(obs)

    def __iter__(self):
        return iter(self.net)


class _Actor(_Net):
    def __init__(self, sizes, act):
        super().__init__(sizes, act)
        self.log_std = torch.nn.Parameter(torch.full((sizes[-1],), math.log(0.5)), requires_grad=False)   # core.py:238-240


class ActorCritic(torch.nn.Module):
    def __init__(self, obs_dim, act_dim=4, pi_hidden=(50, 50), v_hidden=(64, 64), device='cuda',
                 use_standardized_obs=True, use_scaled_rewards=True, dist=None, fused=True, seed=0,
                 policy_kernel='tc'):
        super().__init__()
        # policy_kernel: 'tc' = tcgen05 tensor-core kernel, split-TF32 operands (float32-level results);
        # 'tc_tf32' = the same with operands rounded to TF32 once (~1e-3 relative error on mu / value);
        # 'cuda' = the CUDA-core float32 kernel (also the fallback for shapes the tensor-core plan rejects)
        self.tc_precision = {'tc': 3, 'tc_tf32': 1, 'cuda': 0}[policy_kernel]
        # fused: one CUDA kernel (pdx_policy_step) does standardise + both MLPs + sample + log-prob;
        # the torch modules below stay the owners of the weights (training updates them in place)
        self.fused = (fused and len(pi_hidden) == 2 and len(v_hidden) == 2 and max(*pi_hidden, *v_hidden) <= 64
                      and act_dim <= 4)
        self.seed, self._counter = int(seed), 0
        # global index of row 0 of the observation batches (the collector sets it from its VecEnv): the action
        # noise is keyed by the GLOBAL environment index, so a rollout does not depend on the sharding
        self.env_offset = 0
        self.pi = _Actor([obs_dim, *pi_hidden, act_dim], torch.nn.ReLU)
        self.v = _Net([obs_dim, *v_hidden, 1], torch.nn.Tanh)
        self.to(device)
        self.obs_oms = OnlineMeanStd(obs_dim, device, dist=dist) if use_standardized_obs else None
        self.ret_oms = OnlineMeanStd(1, device, dist=dist) if use_scaled_rewards else None

    @property
    def log_std(self):
        return self.pi.log_std

    def set_log_std(self, frac):                                              # core.py:268-276
        self.pi.log_std.fill_(math.log(0.499 * frac + 0.01))

    # the Philox position of the policy noise is part of a checkpoint (a restored run must not replay draws)
    def get_extra_state(self):
        return {'seed': self.seed, 'counter': self._counter}

    def set_extra_state(self, state):
        self.seed, self._counter = int(state['seed']), int(state['counter'])

    @torch.no_grad()
    def value(self, obs):
        """V(obs) [N].  On CUDA with kernel-supported shapes this is the fused policy kernel (its action
        draw is discarded and does not advance the policy's Philox counter); otherwise the torch modules."""
        if self.fused and obs.is_cuda and obs.dtype == torch.float32 and obs.dim() == 2 and self.log_std.shape[0] == 4:
            n = obs.shape[0]
            scratch = getattr(self, '_value_scratch', None)
            if scratch is None or scratch[0].shape[0] != n or scratch[0].device != obs.device:
                scratch = (torch.empty((n, 4), dtype=torch.float32, device=obs.device),
                           torch.empty(n, dtype=torch.float32, device=obs.device))
                self._value_scratch = scratch
            val = torch.empty(n, dtype=torch.float32, device=obs.device)
            self._launch_into(obs.contiguous(), scratch[0], val, scratch[1], None, counter=0)
            return val
        o = obs.float()
        if self.obs_oms:
            o = self.obs_oms(o)
        return self.v(o).squeeze(-1)

    def _mlp_struct(self, net, n_out):
        lins = [m for m in net if isinstance(m, torch.nn.Linear)]
        st = _lib.PdxMlp()
        st.hidden[0], st.hidden[1], st.n_out = lins[0].out_features, lins[1].out_features, n_out
        for k, lin in enumerate(lins):
            assert lin.weight.is_contiguous() and lin.weight.dtype == torch.float32
            st.weight[k], st.bias[k] = lin.weight.data_ptr(), lin.bias.data_ptr()
        return st

    def _packed_weights(self, obs_dim, pi, v, stream):
        """Device blob of the transposed / padded weights, re-packed when a parameter changed
        (torch bumps `_version` on every in-place update)."""
        params = [p_ for net in (self.pi, self.v) for p_ in net.parameters()]
        L = _lib.load()
        prec = self.tc_precision
        if prec and int(L.pdx_policy_tc_pack_words(obs_dim, C.byref(pi), C.byref(v), prec)) < 0:
            prec = self.tc_precision = 0                  # shapes outside the tensor-core plan
        ver = tuple(p_._version for p_ in params) + tuple(p_.data_ptr() for p_ in params) + (prec,)
        if getattr(self, '_pack_ver', None) != ver:
            words = int(L.pdx_policy_tc_pack_words(obs_dim, C.byref(pi), C.byref(v), prec) if prec
                        else L.pdx_policy_pack_words(obs_dim, C.byref(pi), C.byref(v)))
            if getattr(self, '_pack', None) is None or self._pack.numel() != words:
                self._pack = torch.empty(words, dtype=torch.float32, device=params[0].device)
            if prec:
                _lib.check(L.pdx_policy_tc_pack(obs_dim, C.byref(pi), C.byref(v), prec, C.c_void_p(self._pack.data_ptr()), stream))
            else:
                _lib.check(L.pdx_policy_pack(obs_dim, C.byref(pi), C.byref(v), C.c_void_p(self._pack.data_ptr()), stream))
            self._pack_ver = ver
        return self._pack

    def _launch_policy(self, head, counter, tail, stream, overlap=False):
        """head = (n, d, obs, mean, std, eps, pi, v, log_std, pack, seed); tail = (act, val, logp, mu)."""
        L = _lib.load()
        if self.tc_precision:
            prec = self.tc_precision | (_lib.PDX_POLICY_TC_OVERLAP if overlap else 0)
            return L.pdx_policy_step_tc(*head[:10], prec, head[10], counter, self.env_offset, *tail, stream)
        return L.pdx_policy_step(*head, counter, self.env_offset, *tail, stream)

    @torch.no_grad()
    def step_into(self, obs, act, val, logp, mu=None):
        """Fused ActorCritic.step: obs [N, D] float32 CUDA -> writes act [N, 4], val [N], logp [N]
        (and optionally the Gaussian mean) in ONE kernel launch."""
        assert obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous()
        n, d = obs.shape
        for t in (act, val, logp):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        assert act.shape == (n, 4)
        self._counter += 1
        self._launch_into(obs, act, val, logp, mu, self._counter)

    def _launch_into(self, obs, act, val, logp, mu, counter):
        n, d = obs.shape
        pi, v = self._mlp_struct(self.pi, self.log_std.shape[0]), self._mlp_struct(self.v, 1)
        oms = self.obs_oms
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        st = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
        pack = self._packed_weights(d, pi, v, st)
        head = (n, d, p(obs), p(oms.mean) if oms else None, p(oms.std) if oms else None, oms.eps if oms else 0.0,
                C.byref(pi), C.byref(v), p(self.log_std.data), p(pack), self.seed)
        _lib.check(self._launch_policy(head, counter, (p(act), p(val), p(logp), p(mu)), st))

    def prepare_step_into(self, obs, act, val, logp, overlap=False):
        """Handle for `step_prepared`: all ctypes arguments of one fused policy step, built once.
        overlap: promise that the kernel launched right before each use of the handle writes neither the
        weights nor the normaliser (PDX_POLICY_TC_OVERLAP; tensor-core kernel only).
        Valid while the tensors and the (in place updated) parameters stay where they are."""
        assert obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous() and act.shape == (obs.shape[0], 4)
        pi, v = self._mlp_struct(self.pi, self.log_std.shape[0]), self._mlp_struct(self.v, 1)
        oms = self.obs_oms
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        st = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
        pack = self._packed_weights(obs.shape[1], pi, v, st)
        head = (obs.shape[0], obs.shape[1], p(obs), p(oms.mean) if oms else None, p(oms.std) if oms else None,
                oms.eps if oms else 0.0, C.byref(pi), C.byref(v), p(self.log_std.data), p(pack), self.seed)
        tail = (p(act), p(val), p(logp), None)
        return (head, tail, pi, v, obs, act, val, logp, bool(overlap))

    def refresh_packed_weights(self, obs_dim, stream=None):
        """Call after an optimiser step when prepared handles are in use (the blob keeps its address)."""
        pi, v = self._mlp_struct(self.pi, self.log_std.shape[0]), self._mlp_struct(self.v, 1)
        self._packed_weights(obs_dim, pi, v, stream or C.c_void_p(torch.cuda.current_stream().cuda_stream))

    def step_prepared(self, handle, stream):
        self._counter += 1
        rc = self._launch_policy(handle[0], self._counter, handle[1], stream, handle[8])
        if rc:
            _lib.check(rc)

    @torch.no_grad()
    def step(self, obs, generator=None):
        """obs [N, D] on device -> (action [N, 4], value [N], logp [N]), all on device.  CUDA float32
        observations with kernel-supported shapes always take the fused kernel; the torch expression
        below serves CPU tensors (host-logic tests), explicit generators and wider networks."""
        if self.fused and obs.is_cuda and generator is None and obs.dtype == torch.float32 and self.log_std.shape[0] == 4:
            n = obs.shape[0]
            act = torch.empty((n, 4), dtype=torch.float32, device=obs.device)
            val = torch.empty(n, dtype=torch.float32, device=obs.device)
            logp = torch.empty(n, dtype=torch.float32, device=obs.device)
            self.step_into(obs.contiguous(), act, val, logp)
            return act, val, logp
        o = obs.float()
        if self.obs_oms:
            o = self.obs_oms(o)
        v = self.v(o).squeeze(-1)
        mu = self.pi(o)
        std = torch.exp(self.log_std)
        eps = torch.randn(mu.shape, device=mu.device, dtype=mu.dtype, generator=generator)
        a = mu + std * eps
        logp = (-0.5 * eps ** 2 - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        return a, v, logp


# ---------------------------------------------------------------------------------------------
#  collector
# ---------------------------------------------------------------------------------------------
class RolloutCollector:
    """roll_out() of IWPGAlgorithm for a VecEnv: T lock-step steps of N environments.

    reset_each_rollout=True is the reference's behaviour (the env is reset at the start of every
    roll_out and episodes never span epochs, iwpg.py:353,375); False lets episodes continue."""

    def __init__(self, env, ac, steps, gamma=0.99, lam=0.95, reset_each_rollout=True, dist=None,
                 use_cuda_graphs=True):
        assert env.final_obs is not None, 'construct the VecEnv with keep_final_obs=True'
        self.env, self.ac, self.T, self.gamma, self.lam = env, ac, int(steps), gamma, lam
        self.reset_each_rollout, self.dist = reset_each_rollout, dist
        n, d, dev, T = env.num_envs, env.obs_dim, env.device, self.T
        self.obs = torch.zeros((T + 1, n, d), dtype=env.dtype, device=dev)
        self.act = torch.zeros((T, n, 4), dtype=torch.float32, device=dev)
        self.rew = torch.zeros((T, n), dtype=env.dtype, device=dev)
        self.cost = torch.zeros((T, n), dtype=env.dtype, device=dev)
        self.val = torch.zeros((T, n), dtype=torch.float32, device=dev)
        self.logp = torch.zeros((T, n), dtype=torch.float32, device=dev)
        self.term = torch.zeros((T, n), dtype=torch.uint8, device=dev)
        self.trunc = torch.zeros((T, n), dtype=torch.uint8, device=dev)
        self.boot = torch.zeros((T, n), dtype=torch.float32, device=dev)
        self._outs = [{'obs': self.obs[t + 1], 'reward': self.rew[t], 'cost': self.cost[t],
                       'terminated': self.term[t], 'truncated': self.trunc[t]} for t in range(T)]
        self._started = False
        self.use_cuda_graphs = use_cuda_graphs
        self._graphs = None
        self._prepared = None
        self.ac.env_offset = env.env_offset
        self.last_val = torch.zeros(n, dtype=torch.float32, device=dev)
        self.use_fused_kernel = True           # pdx_collect: policy + env.step of the whole rollout in ONE launch
        self.fused_used = False                # did the last collect() run through pdx_collect?
        self._final_obs_T = None               # [T, N, D], only when truncations can occur inside a rollout
        self._obs_moments = None

    def _fused(self, generator=None):
        return (self.ac.fused and generator is None and self.env.dtype == torch.float32
                and self.ac.log_std.shape[0] == 4)

    def _policy_step(self, t, generator=None):
        if self._fused(generator):
            self.ac.step_into(self.obs[t], self.act[t], self.val[t], self.logp[t])
            return
        a, v, logp = self.ac.step(self.obs[t], generator)
        self.act[t], self.val[t], self.logp[t] = a, v, logp

    def _capture(self):
        """One CUDA graph per step index: obs[t] -> act[t], val[t], logp[t] (normalise, two MLPs,
        sample, log-prob: ~25 small kernels collapse into one graph launch)."""
        cur = torch.cuda.current_stream(self.env.device)
        side = torch.cuda.Stream(self.env.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(3):
                self._policy_step(0)
        cur.wait_stream(side)
        self._graphs, pool = [], None
        for t in range(self.T):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                self._policy_step(t)
            pool = pool or g.pool()
            self._graphs.append(g)

    def _may_truncate(self):
        """Can an episode hit the time limit (or the non-finite guard) inside a rollout?"""
        return (not self.reset_each_rollout) or self.T >= self.env.max_episode_steps or bool(self.env.cfg.reset_on_nonfinite)

    def _collect_fused(self):
        """The whole rollout in ONE launch (pdx_collect): returns False when the configuration is outside the
        fused kernel's plan (the caller then alternates the policy and env.step kernels)."""
        env, ac, T = self.env, self.ac, self.T
        if not (self.use_fused_kernel and ac.tc_precision in (1, 3) and env.rng == 'philox' and env.pdx.observation_noise
                and env.pdx.control_mode == 0 and env.pdx.task != _lib.PDX_TASK['takeoff'] and env.obs_dim % 16 != 0
                and env.obs_dim <= 64 and env.pdx.auto_reset):
            return False
        L = _lib.load()
        p = lambda t: t.data_ptr() if t is not None else None
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        pi, v = ac._mlp_struct(ac.pi, ac.log_std.shape[0]), ac._mlp_struct(ac.v, 1)
        if pi.hidden[0] > 63:                       # the kernel needs room for a constant-1 unit after the actor's first layer
            return False
        pack = ac._packed_weights(env.obs_dim, pi, v, stream)
        if ac.tc_precision not in (1, 3):          # the shapes fell outside the tensor-core plan while packing
            return False
        may_trunc = self._may_truncate()
        if may_trunc and self._final_obs_T is None:
            self._final_obs_T = torch.zeros((T, env.num_envs, env.obs_dim), dtype=env.dtype, device=env.device)
        buf = _lib.PdxBuffers.from_buffer_copy(env._buf)
        buf.obs, buf.reward, buf.cost = p(self.obs[1:]), p(self.rew), p(self.cost)
        buf.terminated, buf.truncated = p(self.term), p(self.trunc)
        buf.final_obs = p(self._final_obs_T) if may_trunc else None
        buf.episode_return = buf.episode_length = None
        oms = ac.obs_oms
        pol = _lib.PdxPolicy()
        pol.obs_dim, pol.precision = env.obs_dim, ac.tc_precision
        pol.mean, pol.std, pol.eps = (p(oms.mean), p(oms.std), oms.eps) if oms is not None else (None, None, 0.0)
        pol.pi, pol.v = C.pointer(pi), C.pointer(v)
        pol.log_std, pol.packed = p(ac.log_std.data), p(pack)
        pol.seed, pol.counter = ac.seed, ac._counter + 1
        out = _lib.PdxRollout()
        out.n_steps, out.obs0 = T, p(self.obs[0])
        out.act, out.val, out.logp, out.last_val = p(self.act), p(self.val), p(self.logp), p(self.last_val)
        if getattr(self, '_scratch', None) is None:
            self._scratch = torch.empty(int(L.pdx_collect_scratch_bytes(env.device.index)), dtype=torch.uint8, device=env.device)
        out.scratch, out.scratch_bytes = p(self._scratch), self._scratch.numel()
        self._obs_moments = None
        if oms is not None:                        # the running-statistics sums of the rollout, accumulated in-kernel
            self._obs_moments = (torch.zeros(2 * env.obs_dim, dtype=torch.float64, device=env.device), oms.mean.clone())
            out.obs_moments = p(self._obs_moments[0])
        rc = L.pdx_collect(C.byref(env.pdx), C.byref(buf), C.byref(pol), C.byref(out), env.seed, env._counter + 1, stream)
        if rc == -1:                               # PDX_ERR_INVALID: outside the fused plan
            return False
        _lib.check(rc)
        env._counter += T
        ac._counter += T
        if may_trunc:
            # time-limit truncations bootstrap with V(last observation of the episode), iwpg.py:371-380: rare
            # (once per max_episode_steps and environment), so they are gathered after the launch
            idx = self.trunc.view(-1).nonzero().squeeze(-1)
            if idx.numel():
                rows = self._final_obs_T.view(T * env.num_envs, -1)[idx].float().contiguous()
                self.boot.view(-1)[idx] = ac.value(rows)
        return True

    def collect(self, generator=None):
        env, ac, T = self.env, self.ac, self.T
        torch.cuda.nvtx.range_push('pdx_collect')
        if self.reset_each_rollout or not self._started:
            self.obs[0].copy_(env.reset())
            self._started = True
        else:
            self.obs[0].copy_(self.obs[T])
        env.clear_episode_stats()
        self.boot.zero_()
        limit = env.max_episode_steps
        fused = self._fused(generator)
        self.fused_used = fused and self._collect_fused()
        if self.fused_used:
            return self._finish(self.last_val)
        graphs = self.use_cuda_graphs and generator is None and not fused
        if graphs and self._graphs is None:
            self._capture()
        if fused and self._prepared is None:
            # inside the loop a policy launch follows an env.step launch and vice versa: neither writes what
            # the other stages before its dependency wait (weights / normaliser; env state), so both may
            # start under the predecessor's tail (programmatic dependent launch).  Measured on B200: with
            # the split-TF32 policy kernel (one 199 KB CTA per SM) early launch of BOTH kernels collapses
            # throughput (0.12 G env-steps/s), early launch of the policy kernel alone gives +5 %.
            early_env = ac.tc_precision != 3
            self._prepared = [(ac.prepare_step_into(self.obs[t], self.act[t], self.val[t], self.logp[t], overlap=t > 0),
                               env.prepare_step(self.act[t], self._outs[t], state_stable=early_env)) for t in range(T)]
        stream = C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)
        if fused:
            ac.refresh_packed_weights(env.obs_dim, stream)
        for t in range(T):
            if fused:                                    # two prepared C-ABI launches per step
                ac.step_prepared(self._prepared[t][0], stream)
                env.step_prepared(self._prepared[t][1], stream)
                if (not self.reset_each_rollout) or t + 1 >= limit or env.cfg.reset_on_nonfinite:
                    self.boot[t] = ac.value(env.final_obs) * self.trunc[t].float()
                continue
            if graphs:
                self._graphs[t].replay()
            else:
                self._policy_step(t, generator)
            env.step(self.act[t], out=self._outs[t])
            # time-limit truncation needs V(last observation of the episode); the engine only
            # truncates when an episode reaches max_episode_steps, i.e. not before step `limit`
            if (not self.reset_each_rollout) or t + 1 >= limit or env.cfg.reset_on_nonfinite:
                self.boot[t] = ac.value(env.final_obs) * self.trunc[t].float()
        self.last_val.copy_(ac.value(self.obs[T]))          # as pdx_collect does: last_val is the cut's bootstrap on both paths
        return self._finish(self.last_val)

    def _finish(self, last_val):
        env, ac, T = self.env, self.ac, self.T
        # iwpg.py:371-380: a time-limit hit bootstraps even if the env also terminated
        done = torch.where(self.trunc > 0, torch.full_like(self.term, 2), self.term)
        ret_std = ac.ret_oms.std if ac.ret_oms is not None else None
        adv, target_v, disc_ret = compute_gae(self.rew, self.val, done, self.boot, last_val, self.gamma,
                                              self.lam, ret_std.data if ret_std is not None else None)
        stats = allreduce_episode_stats(env.episode_stats(), self.dist)
        torch.cuda.nvtx.range_pop()
        return {'obs': self.obs[:T], 'act': self.act, 'adv': adv, 'target_v': target_v, 'log_p': self.logp,
                'discounted_ret': disc_ret, 'rew': self.rew, 'val': self.val, 'done': done,
                'episode_stats': EpisodeStats(stats),
                'obs_moments': self._obs_moments if self.fused_used else None}

    def update_running_statistics(self, data):
        """iwpg.py:387-396: after the update phase, on the raw observations / discounted returns."""
        if self.ac.obs_oms is not None:
            mom = data.get('obs_moments')
            if mom is not None:                    # sums accumulated by pdx_collect: no pass over the observations
                d = self.env.obs_dim
                self.ac.obs_oms.update_from_sums(mom[0][:d], mom[0][d:], self.T * self.env.num_envs, shift=mom[1])
            else:
                self.ac.obs_oms.update(data['obs'])
        if self.ac.ret_oms is not None:
            self.ac.ret_oms.update(data['discounted_ret'].reshape(-1, 1))
