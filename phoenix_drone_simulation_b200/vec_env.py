"""Lock-step vectorised Crazyflie environments on one GPU.

`VecEnv` is the new batched API (absent from the reference): N environments advance with
one fused CUDA kernel launch per `step`, auto-resetting finished episodes inside the same
launch.  Semantics per environment are the reference's `DroneBaseEnv.reset/step`
(envs/base.py:382-475 of phoenix_drone_simulation) -- see csrc/pdx_model.cuh.

All tensors are PyTorch CUDA tensors; the kernels are reached through the C ABI of
libphoenix_b200.so (include/phoenix_b200.h) on torch's current stream.  There is no CPU
path: constructing a VecEnv without a CUDA device raises.
"""
import ctypes as C

import torch

from . import lib as _lib
from .config import EnvConfig


class VecEnv:
    """N environments of one env id, stepped in lock-step on one CUDA device.

    Parameters mirror the reference's `gym.make(env_id, **kwargs)` (config.EnvConfig) plus
      num_envs, device, dtype (torch.float32 throughput mode / torch.float64 parity mode),
      seed (Philox key), env_offset (global index of env 0 of this shard: results do not
      depend on how environments are sharded), rng ('philox' | 'tape'),
      keep_final_obs (also return the last observation of finished episodes).

    With auto_reset=False (config.EnvConfig) a finished environment is not reset in the step: it steps on from its
    terminal state, as the reference does until the caller resets it (`reset(mask)`).  Its episode length keeps
    counting, so `truncated` stays set once the time limit is reached and `terminated` follows done() step by step.
    Every step on which an environment's episode is over (terminated or truncated) counts as a finished episode in
    episode_stats() and reports the running length / return in `episode_length` / `episode_return`: an episode that
    stays ended is counted again on each step.  The reset-package counters (`episode_counters`) do not move.
    """

    def __init__(self, env_id, num_envs, device='cuda', dtype=torch.float32, seed=0,
                 env_offset=0, rng='philox', keep_final_obs=False, **kwargs):
        if not torch.cuda.is_available():
            raise _lib.PhoenixB200Error('VecEnv needs a CUDA device: there is no CPU fallback')
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.PhoenixB200Error('VecEnv needs a CUDA device: there is no CPU fallback')
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        if dtype not in (torch.float32, torch.float64):
            raise ValueError('dtype must be torch.float32 or torch.float64')
        self.dtype = dtype
        self.num_envs = int(num_envs)
        self.env_id = env_id
        self.cfg = kwargs.pop('config', None) or EnvConfig(env_id, **kwargs)
        self.rng = rng
        self.pdx = self.cfg.to_pdx(
            _lib.PDX_DTYPE_F32 if dtype == torch.float32 else _lib.PDX_DTYPE_F64,
            _lib.PDX_RNG_PHILOX if rng == 'philox' else _lib.PDX_RNG_TAPE)
        self.obs_dim = int(self.pdx.obs_dim)
        self.core_dim = int(self.pdx.core_dim)
        self.act_dim = 4
        self.max_episode_steps = int(self.pdx.max_episode_steps)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.env_offset = int(env_offset)
        self._counter = 0
        n, dev = self.num_envs, self.device
        self.n_quads = self.lib.pdx_state_quads(C.byref(self.pdx))
        self.state = torch.zeros((self.n_quads, n, 4), dtype=dtype, device=dev)
        self.obs = torch.zeros((n, self.obs_dim), dtype=dtype, device=dev)
        self.reward = torch.zeros(n, dtype=dtype, device=dev)
        self.cost = torch.zeros(n, dtype=dtype, device=dev)
        self._terminated = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.terminated = self._terminated.view(torch.bool)
        self.truncated = self._truncated.view(torch.bool)
        self.episode_return = torch.zeros(n, dtype=dtype, device=dev)
        self.episode_length = torch.zeros(n, dtype=torch.int32, device=dev)
        self.final_obs = torch.zeros((n, self.obs_dim), dtype=dtype, device=dev) if keep_final_obs else None
        self.stats = torch.zeros(8, dtype=torch.float64, device=dev)
        self.clear_episode_stats()
        rs, ss, is_ = C.c_int(), C.c_int(), C.c_int()
        self.lib.pdx_tape_slots(C.byref(self.pdx), C.byref(rs), C.byref(ss), C.byref(is_))
        self.tape_slots = dict(reset=rs.value, step=ss.value, init=is_.value)
        self._tapes = dict(step=None, reset=None, init=None)
        self.step_bytes = int(self.lib.pdx_step_bytes(C.byref(self.pdx)))
        self._buf = _lib.PdxBuffers()
        self._fill_buffers()
        if rng == 'philox':
            self._construct()

    # ----------------------------------------------------------------------------------------
    def _fill_buffers(self):
        b = self._buf
        b.n_envs, b.env_offset, b.device = self.num_envs, self.env_offset, self.device.index
        b.state, b.obs = self.state.data_ptr(), self.obs.data_ptr()
        b.reward, b.cost = self.reward.data_ptr(), self.cost.data_ptr()
        b.terminated, b.truncated = self._terminated.data_ptr(), self._truncated.data_ptr()
        b.final_obs = self.final_obs.data_ptr() if self.final_obs is not None else None
        b.episode_return = self.episode_return.data_ptr()
        b.episode_length = self.episode_length.data_ptr()
        b.episode_stats = self.stats.data_ptr()
        for k in ('step', 'reset', 'init'):
            t = self._tapes[k]
            setattr(b, 'tape_' + k, t.data_ptr() if t is not None else None)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _next_counter(self):
        self._counter += 1
        return self._counter

    def _construct(self):
        """Constructor semantics of the reference (state zeroed, nominal parameters, the one
        compute_observation() call of base.py:143)."""
        _lib.check(self.lib.pdx_init(C.byref(self.pdx), C.byref(self._buf), self.seed, 0, self._stream()))

    # ---- tape mode (parity harness) ---------------------------------------------------------
    def set_tapes(self, step=None, reset=None, init=None):
        """Standardised draws, float64 CUDA tensors of shape [slots, num_envs]."""
        for k, t in (('step', step), ('reset', reset), ('init', init)):
            if t is not None:
                assert t.dtype == torch.float64 and t.is_cuda and t.is_contiguous()
                assert t.shape == (self.tape_slots[k], self.num_envs), (k, tuple(t.shape), self.tape_slots[k])
                self._tapes[k] = t
        self._fill_buffers()

    def construct_from_tape(self, init=None):
        if init is not None:
            self.set_tapes(init=init)
        self._construct()

    # ---- API ------------------------------------------------------------------------------
    def reset(self, mask=None):
        """Reset all environments (or those where `mask` is True); returns obs [N, D]."""
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mptr = C.c_void_p(mask.data_ptr())
        _lib.check(self.lib.pdx_reset(C.byref(self.pdx), C.byref(self._buf), mptr, self.seed,
                                      self._next_counter(), self._stream()))
        return self.obs

    def step(self, actions, out=None):
        """actions: float32 CUDA tensor [N, 4].  Returns (obs, reward, terminated, truncated,
        info); the tensors are owned by the VecEnv and overwritten by the next call.

        `out` (optional): dict of caller-owned CUDA tensors that receive this step's results
        instead -- keys 'obs' [N, D], 'reward' [N], 'cost' [N] (engine dtype), 'terminated' [N],
        'truncated' [N] (uint8); missing keys fall back to the VecEnv's own buffers.  This is how
        the rollout collector stores straight into its [T, N, .] tensors."""
        if actions.dtype != torch.float32 or not actions.is_contiguous() or actions.device != self.device:
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        assert actions.shape == (self.num_envs, 4)
        buf = self._buf
        if out:
            buf = _lib.PdxBuffers.from_buffer_copy(self._buf)
            for k, t in out.items():
                assert t.is_cuda and t.is_contiguous() and t.shape[0] == self.num_envs, k
                setattr(buf, k, t.data_ptr())
        _lib.check(self.lib.pdx_step(C.byref(self.pdx), C.byref(buf), C.c_void_p(actions.data_ptr()),
                                     self.seed, self._next_counter(), self._stream()))
        if out:
            return (out.get('obs', self.obs), out.get('reward', self.reward),
                    out['terminated'].view(torch.bool) if 'terminated' in out else self.terminated,
                    out['truncated'].view(torch.bool) if 'truncated' in out else self.truncated,
                    {'cost': out.get('cost', self.cost), 'episode_return': self.episode_return,
                     'episode_length': self.episode_length})
        info = {'cost': self.cost, 'episode_return': self.episode_return,
                'episode_length': self.episode_length}
        if self.final_obs is not None:
            info['final_observation'] = self.final_obs
        return self.obs, self.reward, self.terminated, self.truncated, info

    # ---- prepared launches: everything that does not change between calls is built once ------
    def prepare_step(self, actions, out, state_stable=False):
        """Returns a handle for `step_prepared`: the PdxBuffers of a step that reads `actions`
        [N, 4] and writes into the tensors of `out` (see `step`).  The tensors must stay alive.
        state_stable: promise that the kernel launched right before each use of this handle does not
        write this VecEnv's state (PDX_BUF_STATE_STABLE: the state load overlaps that kernel's tail)."""
        assert actions.dtype == torch.float32 and actions.is_contiguous() and actions.shape == (self.num_envs, 4)
        buf = _lib.PdxBuffers.from_buffer_copy(self._buf)
        for k, t in out.items():
            assert t.is_cuda and t.is_contiguous() and t.shape[0] == self.num_envs, k
            setattr(buf, k, t.data_ptr())
        if state_stable:
            buf.flags |= _lib.PDX_BUF_STATE_STABLE
        return (C.byref(self.pdx), C.byref(buf), C.c_void_p(actions.data_ptr()), buf, actions, out)

    def step_prepared(self, handle, stream):
        """`stream`: C.c_void_p of the CUDA stream (cache it: looking it up costs microseconds)."""
        self._counter += 1
        rc = self.lib.pdx_step(handle[0], handle[1], handle[2], self.seed, self._counter, stream)
        if rc:
            _lib.check(rc)

    def step_many(self, actions, out):
        """T env.steps of every environment in ONE kernel launch (state stays in registers
        between steps; open-loop action sequence).  actions: float32 CUDA tensor [T, N, 4];
        `out`: dict of time-major CUDA tensors -- 'obs' [T, N, D], 'reward', 'cost' [T, N] (engine
        dtype), 'terminated', 'truncated' [T, N] (uint8); optional 'final_obs' [T, N, D],
        'episode_return' [T, N], 'episode_length' [T, N] (int32).  Returns `out`."""
        assert actions.dtype == torch.float32 and actions.is_contiguous() and actions.device == self.device
        T = actions.shape[0]
        assert actions.shape == (T, self.num_envs, 4)
        buf = _lib.PdxBuffers.from_buffer_copy(self._buf)
        buf.final_obs = buf.episode_return = buf.episode_length = None
        for k in ('obs', 'reward', 'cost', 'terminated', 'truncated'):
            assert k in out, k
        for k, t in out.items():
            assert t.is_cuda and t.is_contiguous() and t.shape[0] == T and t.shape[1] == self.num_envs, k
            setattr(buf, k, t.data_ptr())
        assert self.rng == 'philox', 'step_many draws on device'
        torch.cuda.nvtx.range_push('pdx_step_many')         # shows up in nsys / ncu --nvtx timelines
        _lib.check(self.lib.pdx_step_many(C.byref(self.pdx), C.byref(buf), C.c_void_p(actions.data_ptr()), T,
                                          self.seed, self._counter + 1, self._stream()))
        torch.cuda.nvtx.range_pop()
        self._counter += T
        return out

    def make_host_pipeline(self, n_steps, chunk_steps=8):
        """Pinned host buffers + double-buffered device staging for `step_many_host`."""
        T, c, n, d = int(n_steps), int(chunk_steps), self.num_envs, self.obs_dim
        assert T % c == 0
        dev, dt = self.device, self.dtype
        pin = lambda *shape, dtype: torch.empty(shape, dtype=dtype).pin_memory()
        host = {'actions': pin(T, n, 4, dtype=torch.float32), 'obs': pin(T, n, d, dtype=dt),
                'reward': pin(T, n, dtype=dt), 'cost': pin(T, n, dtype=dt),
                'terminated': pin(T, n, dtype=torch.uint8), 'truncated': pin(T, n, dtype=torch.uint8)}
        stage = [{'actions': torch.empty((c, n, 4), dtype=torch.float32, device=dev),
                  'obs': torch.empty((c, n, d), dtype=dt, device=dev),
                  'reward': torch.empty((c, n), dtype=dt, device=dev), 'cost': torch.empty((c, n), dtype=dt, device=dev),
                  'terminated': torch.empty((c, n), dtype=torch.uint8, device=dev),
                  'truncated': torch.empty((c, n), dtype=torch.uint8, device=dev)} for _ in range(2)]
        streams = [torch.cuda.Stream(dev) for _ in range(3)]
        h2d_bytes = host['actions'].numel() * 4
        d2h_bytes = sum(host[k].numel() * host[k].element_size() for k in host if k != 'actions')
        return {'host': host, 'stage': stage, 'streams': streams, 'T': T, 'chunk': c,
                'h2d_bytes': h2d_bytes, 'd2h_bytes': d2h_bytes}

    def step_many_host(self, pipe):
        """T env.steps with HOST action / result buffers (pipe['host'], pinned): the actions of
        chunk k+1 travel host->device and the results of chunk k-1 device->host while chunk k
        computes (three streams, two staging sets).  Returns after the copies are enqueued; the
        caller synchronises (or records an event on the current stream, which waits for them)."""
        host, stage, (s_in, s_run, s_out) = pipe['host'], pipe['stage'], pipe['streams']
        T, c = pipe['T'], pipe['chunk']
        cur = torch.cuda.current_stream(self.device)
        for s in (s_in, s_run, s_out):
            s.wait_stream(cur)
        ev_in, ev_run, ev_out = {}, {}, {}
        outs = ('obs', 'reward', 'cost', 'terminated', 'truncated')
        for k in range(T // c):
            st = stage[k & 1]
            with torch.cuda.stream(s_in):
                if k >= 2:
                    s_in.wait_event(ev_run[k - 2])          # staging actions consumed
                st['actions'].copy_(host['actions'][k * c:(k + 1) * c], non_blocking=True)
                ev_in[k] = s_in.record_event()
            with torch.cuda.stream(s_run):
                s_run.wait_event(ev_in[k])
                if k >= 2:
                    s_run.wait_event(ev_out[k - 2])         # staging results drained
                self.step_many(st['actions'], {o: st[o] for o in outs})
                ev_run[k] = s_run.record_event()
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_run[k])
                for o in outs:
                    host[o][k * c:(k + 1) * c].copy_(st[o], non_blocking=True)
                ev_out[k] = s_out.record_event()
        for s in (s_in, s_run, s_out):
            cur.wait_stream(s)
        return host

    def rollout_bytes(self, n_steps):
        """Algorithmic HBM bytes per environment of one n_steps launch (pdx_rollout_bytes)."""
        return int(self.lib.pdx_rollout_bytes(C.byref(self.pdx), int(n_steps)))

    # ---- validation: production Philox draws copied out in tape layout ------------------------
    def dump_init(self):
        t = torch.zeros((max(self.tape_slots['init'], 1), self.num_envs), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pdx_dump_draws(C.byref(self.pdx), C.byref(self._buf), None, self.seed, 0,
                                           None, None, C.c_void_p(t.data_ptr()), self._stream()))
        return t[:self.tape_slots['init']]

    def dump_reset(self):
        t = torch.zeros((max(self.tape_slots['reset'], 1), self.num_envs), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.pdx_dump_draws(C.byref(self.pdx), C.byref(self._buf), None, self.seed,
                                           self._next_counter(), None, C.c_void_p(t.data_ptr()), None,
                                           self._stream()))
        return self.obs, t[:self.tape_slots['reset']]

    def dump_step(self, actions):
        ts = torch.zeros((max(self.tape_slots['step'], 1), self.num_envs), dtype=torch.float64, device=self.device)
        tr = torch.zeros((max(self.tape_slots['reset'], 1), self.num_envs), dtype=torch.float64, device=self.device)
        actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        _lib.check(self.lib.pdx_dump_draws(C.byref(self.pdx), C.byref(self._buf), C.c_void_p(actions.data_ptr()),
                                           self.seed, self._next_counter(), C.c_void_p(ts.data_ptr()),
                                           C.c_void_p(tr.data_ptr()), None, self._stream()))
        return ts[:self.tape_slots['step']], tr[:self.tape_slots['reset']]

    # ---- episode statistics (block-reduced in the step kernel) ------------------------------
    def clear_episode_stats(self):
        if getattr(self, '_stats_init', None) is None:       # device-resident constant: no H2D copy per clear
            self._stats_init = torch.tensor([0., 0., 0., 0., 1e300, -1e300, 1e300, -1e300], dtype=torch.float64,
                                            device=self.stats.device)
        self.stats.copy_(self._stats_init)

    def episode_stats(self, clear=False):
        """[n, sum ret, sum ret^2, sum len, min ret, max ret, min len, max len] (float64)."""
        s = self.stats.clone()
        if clear:
            self.clear_episode_stats()
        return s

    # ---- state access (checkpointing, parity harness) ------------------------------------------
    def _field(self, name):
        fw, nw = C.c_int(), C.c_int()
        _lib.check(self.lib.pdx_state_field(C.byref(self.pdx), name.encode(), C.byref(fw), C.byref(nw)))
        return fw.value, nw.value

    def get_state(self, name):
        fw, nw = self._field(name)
        return torch.stack([self.state[w // 4, :, w % 4] for w in range(fw, fw + nw)], dim=1)

    def set_state(self, name, value):
        fw, nw = self._field(name)
        value = torch.as_tensor(value, dtype=self.dtype, device=self.device).reshape(-1, nw)
        value = value.expand(self.num_envs, nw)
        for k, w in enumerate(range(fw, fw + nw)):
            self.state[w // 4, :, w % 4] = value[:, k]

    def _ep_word(self):
        """The state word ep_index of every environment, a view: uint32 (e << 4) | pend, held as the
        value in float64 and as the bit pattern in float32 (csrc/pdx_layout.h)."""
        fw, _ = self._field('ep_index')
        if self.dtype == torch.float32:
            return self.state.view(torch.int32)[fw // 4, :, fw % 4]
        return self.state[fw // 4, :, fw % 4]

    def episode_counters(self):
        """(episodes, pending): int64 [N] in-kernel auto-resets each environment has consumed, modulo 2^28
        (they key the reset draws), and int32 [N] bit mask of reset-package slots waiting to be regenerated."""
        w = self._ep_word().to(torch.int64) & 0xFFFFFFFF
        return w >> 4, (w & 15).to(torch.int32)

    def set_episode_counters(self, episodes, pending=0b1111):
        """Sets the counters `episode_counters` reports (scalars or [N] tensors; episodes modulo 2^28).
        The pooled packages were drawn for the old counter: with all four pending bits (the default) the
        end of the next step regenerates them under the new keys.  An episode that ends in that first step
        still takes the old package of its slot."""
        e = torch.as_tensor(episodes, dtype=torch.int64, device=self.device) & ((1 << 28) - 1)
        p = torch.as_tensor(pending, dtype=torch.int64, device=self.device)
        assert bool(((p >= 0) & (p < 16)).all()), 'pending is a mask of the 4 package slots'
        w = ((e << 4) | p).expand(self.num_envs)
        if self.dtype == torch.float32:
            w = torch.where(w >= 1 << 31, w - (1 << 32), w).to(torch.int32)   # the same 32 bits, as int32
        self._ep_word().copy_(w.to(self._ep_word().dtype))

    def state_dict(self):
        return {'state': self.state.clone(), 'counter': self._counter, 'seed': self.seed,
                'env_id': self.env_id, 'stats': self.stats.clone()}

    def load_state_dict(self, sd):
        assert sd['env_id'] == self.env_id and sd['state'].shape == self.state.shape
        self.state.copy_(sd['state'])
        self.stats.copy_(sd['stats'])
        self._counter = int(sd['counter'])
        self.seed = int(sd['seed'])
