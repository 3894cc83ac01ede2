// Kernels: init (constructor), reset (masked) and the fused multi-step rollout kernel.
//
// k_rollout advances every environment by n_steps env.steps in ONE launch:
//   * one thread owns one environment; its state quads are loaded once (coalesced 128-bit
//     accesses), live in registers across all steps and sub-steps, and are stored once;
//   * each step's observation rows are assembled in a shared-memory tile that has exactly the
//     layout of the block's slice of the row-major [n_envs][obs_dim] output, and leave the SM
//     as ONE bulk asynchronous copy (cp.async.bulk shared->global, the TMA engine; SASS UBLKCP)
//     issued by one thread, double buffered so the copy of step t overlaps step t+1;
//   * episodes that end are reset inside the same launch.  The reset path is as long as a step
//     (two noisy observation calls, ~20 Philox calls) and only a few lanes of a warp need it, so
//     the warp generates the random draws of its finished environments together (shared table,
//     one Philox call per lane and pass) and only the arithmetic runs on the owner lanes;
//   * episode statistics accumulate per thread in shared memory and are reduced once per launch
//     (warp shuffles, one set of atomics per block).
#pragma once
#include "pdx_model.cuh"

namespace pdx {

constexpr int kMaxBlock = 512;     // threads per block are chosen at run time (<= kMaxBlock)

template <class T>
struct KArgs {
  DevCfg<T> c;
  PdxBuffers b;
  const float* actions;
  const uint8_t* mask;
  uint64_t seed, counter;
  double* dump_step;
  double* dump_reset;
  double* dump_init;
  int n_steps;
  int n_tiles;      // 2: observation tiles double buffered; 1: one tile, shifted in place
};

// The ep_index word (pdx_layout.h): uint32_t (e << 4) | pend.  float64 keeps the integer's value (exact below
// 2^53), float32 the bit pattern: a float value would stop holding 16 e + pend exactly at e = 2^20 and lose
// pending bits.  e counts modulo 2^28 (kEpMask) everywhere: here, in the package keys and in the tape path.
__device__ __forceinline__ uint32_t ep_word(const float& w) { return __float_as_uint(w); }
__device__ __forceinline__ uint32_t ep_word(const double& w) { return (uint32_t)w; }
__device__ __forceinline__ void set_ep_word(float& w, uint32_t v) { w = __uint_as_float(v); }
__device__ __forceinline__ void set_ep_word(double& w, uint32_t v) { w = (double)v; }

// `package`: the draws of in-kernel auto-reset number `counter` of this environment (a stream of its
// own: an explicit pdx_reset at call counter c and auto-reset package c must not share draws)
template <class T, int RNG>
__device__ __forceinline__ Rng<T, RNG> make_rng(const KArgs<T>& a, uint64_t counter, int64_t i,
                                                const double* tape, double* dump, bool package = false) {
  Rng<T, RNG> r;
  const uint64_t env = (uint64_t)(a.b.env_offset + i);
  r.key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  r.env_lo = (uint32_t)env;
  r.env_hi = (uint32_t)(env >> 32) ^ ((uint32_t)(counter >> 32) << 8) ^ (package ? 0x80000000u : 0u);
  r.ctr_lo = (uint32_t)counter;
  r.tape = tape ? tape + i : nullptr;
  r.stride = a.b.n_envs;
  r.dump = dump ? dump + i : nullptr;
  return r;
}

// float32 quantisation of the initial position (quirk A.6-6: `pos` is a float32 array)
template <class T> __device__ __forceinline__ T f32q(T x) { return (T)(float)x; }
template <class T> __device__ __forceinline__ T unif(T lo, T hi, T u) { return lo + (hi - lo) * u; }

// ---------------------------------------------------------------------------------------------
//  DroneBaseEnv.reset for one env (base.py:382-431).  `m` holds the state to reset: only the
//  gyro bias (and, for the caller, the OU state) survive a reset (quirk A.6-8); `stale` are the
//  body rates of the previous episode's last state (base.py:411, quirk A.6-5).
//  Outputs: m.w (complete new state, OU words untouched), o1 / o2 = the two observation calls
//  (base.py:420,429); the history is H-1 copies of (o1, last_action) and one (o2, last_action).
// ---------------------------------------------------------------------------------------------
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID, class RG>
__device__ __forceinline__ void reset_env(Model<T, TASK, PHYS, NOISE, RNG, PID>& m, const RG& rng,
                                          const T stale[3], T* o1, T* o2) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  const DevCfg<T>& c = m.c;
  T* w = m.w;
  const T pi = T(3.14159265358979323846);

  T la[4] = {T(0), T(0), T(0), T(0)};                    // drone.last_action = ring[-1]
  T ring[8] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  T x[4] = {T(0), T(0), T(0), T(0)};
  T pos[3] = {c.init_xyz[0], c.init_xyz[1], c.init_xyz[2]};
  T q[4] = {T(0), T(0), T(0), T(1)};
  T vel[3] = {T(0), T(0), T(0)};
  T oms[3] = {T(0), T(0), T(0)};
  T rpy0[3] = {T(0), T(0), T(0)};                        // Euler angles the pose is built from
  int ref_off = 0;
  if constexpr (TASK == PDX_TASK_CIRCLE) ref_off = (int)w[L.ref_offset];

  if constexpr (TASK == PDX_TASK_TAKEOFF) {                        // takeoff.py:179-212
    if (c.reset_distribution) {
      T u[3];
      rng.template uniforms<3>(SITE_RESET, 0, u);
      pos[0] = f32q(pos[0] + unif(T(-0.25), T(0.25), u[0]));
      pos[1] = f32q(pos[1] + unif(T(-0.25), T(0.25), u[1]));
      rpy0[2] = unif(-pi, pi, u[2]);
      quat_from_euler(T(0), T(0), rpy0[2], q);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) { la[k] = T(-1); ring[k] = T(-1); ring[4 + k] = T(-1); }
  } else if (c.reset_distribution) {
    T u[14];
    rng.template uniforms<14>(SITE_RESET, 0, u);
    T rpy[3];
    if constexpr (TASK == PDX_TASK_HOVER) {                        // hover.py:192-229
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        pos[k] = f32q(pos[k] + unif(T(-0.25), T(0.25), u[k]));
        rpy[k] = unif(-(pi / T(6)), pi / T(6), u[3 + k]);
        vel[k] = T(0) + unif(T(-0.1), T(0.1), u[7 + k]);
        const T lim = pi * T(200) / T(180);
        oms[k] = T(0) + unif(-lim, lim, u[10 + k]);
      }
      rpy[2] = unif(-(T(2) * pi), T(2) * pi, u[6]);
    } else {                                             // circle.py:213-256
      // np.random.randint(0, 300): the tape holds the integer itself; Philox: floor(300 u)
      const bool from_tape = RG::kTape && !rng.dumping();
      ref_off = from_tape ? (int)u[0] : min(299, (int)(u[0] * T(300)));
      rng.dump_value(0, (double)ref_off);
      T tp[3];
      m.ref_point(ref_off, tp);
      const T a0 = pi * T(20) / T(180), lim = pi * T(50) / T(180);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        pos[k] = tp[k] + unif(T(-0.05), T(0.05), u[1 + k]);
        rpy[k] = unif(-a0, a0, u[4 + k]);
        vel[k] = T(0) + unif(T(-0.1), T(0.1), u[8 + k]);
      }
      rpy[2] = unif(-(T(0.1) * pi), T(0.1) * pi, u[7]);
      oms[0] = unif(-lim, lim, u[11]);
      oms[1] = unif(-lim, lim, u[12]);
    }
    const T yl = pi * T(20) / T(180);
    oms[2] = unif(-yl, yl, u[13]);
    quat_from_euler(rpy[0], rpy[1], rpy[2], q);
#pragma unroll
    for (int k = 0; k < 3; ++k) rpy0[k] = rpy[k];
    T z[8];
    rng.template normals<8>(SITE_RESET + 4, 14, z);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      x[k] = c.hover_x + T(0.02) * z[k];
      ring[k] = clampT(c.hover_action + T(0.02) * z[4 + k], T(-1), T(1));
    }
    if (c.buf_size > 1) {
      rng.template normals<4>(SITE_RESET + 6, 22, z);
#pragma unroll
      for (int k = 0; k < 4; ++k) ring[4 + k] = clampT(c.hover_action + T(0.02) * z[k], T(-1), T(1));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) la[k] = c.buf_size > 1 ? ring[4 + k] : ring[k];
  }

  // pose / velocity hand-over through "PyBullet": hover.py:232-243, agents.py:434-453
  T R[9];
  rot_from_quat(q, R);
  T ww[3], ob[3];
  ww[0] = R[0] * oms[0] + R[3] * oms[1] + R[6] * oms[2];   // R^T w written as WORLD rate
  ww[1] = R[1] * oms[0] + R[4] * oms[1] + R[7] * oms[2];
  ww[2] = R[2] * oms[0] + R[5] * oms[1] + R[8] * oms[2];
  ob[0] = R[0] * ww[0] + R[3] * ww[1] + R[6] * ww[2];      // ... and R^T again (quirk A.6-4)
  ob[1] = R[1] * ww[0] + R[4] * ww[1] + R[7] * ww[2];
  ob[2] = R[2] * ww[0] + R[5] * ww[1] + R[8] * ww[2];

  // apply_domain_randomization: base.py:239-296, agents.py:208-224
  int slot = c.slots_reset_task;
  if (c.dr_on) {
    auto draw = [&](T v, T uu) { const T b = c.dr * v; return unif(v - b, v + b, uu); };
    T u[15];
    if (Mo::BULLET && c.use_motor_dynamics) rng.template uniforms<15>(SITE_DR, slot, u);
    else rng.template uniforms<7>(SITE_DR, slot, u);
    w[L.dt] = draw(c.time_step, u[0]);
    w[L.mass] = draw(c.mass, u[1]);
    w[L.inertia] = draw(c.inertia[0], u[2]);
    w[L.inertia + 1] = draw(c.inertia[1], u[3]);
    w[L.inertia + 2] = draw(c.inertia[2], u[4]);           // u[5]: ftf0 (cancels, unused)
    w[L.ftf1] = draw(c.ftf1, u[6]);
    if constexpr (Mo::BULLET) if (c.use_motor_dynamics) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const T Tm = M<T>::fmax(draw(c.motor_tc, u[7 + k]), w[L.dt]);
        w[L.motor_b + k] = w[L.dt] / Tm;
        w[L.motor_k + k] = c.k_mass_dr * c.gravity * draw(c.thrust2weight, u[11 + k]) / T(4);  // quirk A.6-7
      }
    }
  }
  slot += c.slots_reset_dr;

  // commit kinematics
#pragma unroll
  for (int k = 0; k < 3; ++k) { w[L.xyz + k] = pos[k]; w[L.vel + k] = vel[k]; }
  if constexpr (Mo::BULLET) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { w[L.quat + k] = q[k]; w[L.motor_x + k] = x[k]; w[L.ring + k] = ring[k]; w[L.ring + 4 + k] = ring[4 + k]; }
#pragma unroll
    for (int k = 0; k < 3; ++k) w[L.omega_world + k] = ww[k];
    w[L.ring_idx] = T(0);
  } else {
    // agents.py:446: rpy = getEulerFromQuaternion(q).  With |roll|, |pitch| < pi/2 (all reset
    // distributions) that round trip is the identity up to wrapping yaw into (-pi, pi]; the
    // float32 kernels use that, the float64 kernels do the reference's round trip.
    T e[3];
    if constexpr (sizeof(T) == 4) {
      e[0] = rpy0[0]; e[1] = rpy0[1];
      e[2] = rpy0[2] - T(6.283185307179586) * rintf(rpy0[2] * T(0.15915494309189535));
    } else {
      euler_from_quat(q, e);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { w[L.rpy + k] = e[k]; w[L.omega + k] = ob[k]; }
  }
  if constexpr (NOISE) {
#pragma unroll
    for (int k = 0; k < 3; ++k) w[L.gyro_lpf + k] = stale[k];
  }
  if constexpr (TASK == PDX_TASK_CIRCLE) w[L.ref_offset] = (T)ref_off;
#pragma unroll
  for (int k = 0; k < 4; ++k) w[L.last_action + k] = la[k];
  w[L.ep_return] = T(0);
  w[L.ep_length] = T(0);
  if constexpr (PID) {                                    // control.reset(): control.py:182-191,282-287
#pragma unroll
    for (int k = 0; k < 12; ++k) w[L.pid + k] = T(0);
  }

  // two observation calls (base.py:420,429)
  T target[3] = {c.target[0], c.target[1], c.target[2]};
  if constexpr (TASK == PDX_TASK_CIRCLE) m.ref_point(ref_off % 300, target);
  if constexpr (TASK == PDX_TASK_TAKEOFF) m.ref_point(0, target);
  m.observe(rng, SITE_RESET_OBS1, slot, target, la, q, o1);
  m.observe(rng, SITE_RESET_OBS2, slot + c.slots_obs_full, target, la, q, o2);
}

// history slots of the state <- H-1 entries, `entry(s, idx)` gives word idx of slot s
template <class T, int E, int QH, class F>
__device__ __forceinline__ void store_history(T* state, int64_t n, int64_t i, int first_quad, int H, F entry) {
  for (int s = 0; s < H - 1; ++s) {
#pragma unroll
    for (int qd = 0; qd < QH; ++qd) {
      T v[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const int idx = qd * 4 + l;
        v[l] = idx < E ? entry(s, idx < E ? idx : 0) : T(0);
      }
      store_quad(state, n, i, first_quad + s * QH + qd, v);
    }
  }
}

// ---------------------------------------------------------------------------------------------
//  Pre-computed reset packages (production Philox path).
//
//  An env.reset() is as long as an env.step (two noisy observation calls, ~20 Philox calls, three
//  Euler->quaternion conversions), and with U(-1,1) actions 11 % of the environments finish per step:
//  3.6 of a warp's 32 lanes.  Running the reset where it happens executes all of it at 11 % lane
//  occupancy, every step.  Nothing in a reset depends on the episode that just ended except three
//  carried words (gyro bias, the stale body rates that seed the low pass: quirks A.6-5 / A.6-8) and
//  those enter LINEARLY.  So the reset of episode p of environment j is keyed by (seed, j, p) -- not
//  by the step at which it happens -- and computed ahead of time:
//    * every environment owns kPackSlots package slots behind its history slots in `state`; slot p & 3 holds
//      the complete state of a freshly reset environment plus its two reset observations, computed
//      with zero carried words (reset_env below, unchanged);
//    * a lane whose episode ends LOADS its package (divergent, but ~16 128-bit loads and a dozen
//      FMAs for the carried words instead of ~500 instructions) and marks the slot pending;
//    * when a warp has 32 pending slots, its 32 lanes regenerate them together, one package per lane,
//      fully converged.  The pending bits live in the state, so when that happens depends only on the
//      history of the 32 environments, not on how the steps are split over launches.
//  The tape (parity) instantiation keeps the in-thread reset; in dump mode it draws with the same
//  (seed, j, p) keys, so pdx_dump_draws reports exactly the draws a package was built from.
// ---------------------------------------------------------------------------------------------
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__device__ __forceinline__ void init_nominal(Model<T, TASK, PHYS, NOISE, RNG, PID>& m) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  const DevCfg<T>& c = m.c;
#pragma unroll
  for (int k = 0; k < Mo::NW; ++k) m.w[k] = T(0);
  m.w[L.xyz + 2] = T(1);                                  // agents.py:32
  m.w[L.dt] = c.time_step;
  m.w[L.mass] = c.mass;
#pragma unroll
  for (int k = 0; k < 3; ++k) m.w[L.inertia + k] = c.inertia[k];
  m.w[L.ftf1] = c.ftf1;
  if constexpr (Mo::BULLET) {
    m.w[L.quat + 3] = T(1);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      m.w[L.motor_b + k] = T(1) * c.time_step / c.motor_tc;   // agents.py:203-204
      m.w[L.motor_k + k] = c.max_thrust;                      // agents.py:200
    }
  }
}

// first plane of the package pool in the state tensor.  The pool region holds kPackSlots * pack_quads planes
// worth of memory but is laid out per package: quad q of the package in slot s of environment j sits at
//   state + ((pool_plane * n + (s * n + j) * pack_quads + q) * 4 reals
// i.e. one package is pack_quads * 16 contiguous bytes (two or three cache lines: a finished lane
// fetches it with a few 128-bit loads of the same lines, and can prefetch it).
template <class Mo>
__device__ __forceinline__ int pool_plane(int history) {
  return Mo::L.n_quads + (history - 1) * Mo::QH;
}
template <class Mo, class T>
__device__ __forceinline__ T* package_ptr(T* state, int64_t n, int64_t j, int history, int slot) {
  const int n32 = (int)n;                                // n < 2^31 (checked at the ABI): 32 x 32 -> 64 bit products
  return state + (((int64_t)pool_plane<Mo>(history) * n32 + ((int64_t)slot * n32 + j) * Mo::L.pack_quads) << 2);
}
template <class T> __device__ __forceinline__ void load_quad_at(const T* p, int q, T* out) { load_quad(p, (int64_t)0, (int64_t)q, 0, out); }
template <class T> __device__ __forceinline__ void store_quad_at(T* p, int q, const T* in) { store_quad(p, (int64_t)0, (int64_t)q, 0, in); }

// package p of environment j (local index) -> its slot.  Zero carried words: the consumer adds their
// (linear) contribution.
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__device__ __forceinline__ void gen_package(const KArgs<T>& a, int64_t j, uint32_t p) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  constexpr int C = Mo::C;
  Mo g(a.c);
  init_nominal(g);
  const Rng<T, RNG> rng = make_rng<T, RNG>(a, (uint64_t)p, j, nullptr, nullptr, true);
  const T stale[3] = {T(0), T(0), T(0)};
  T o1[C], o2[C];
  reset_env(g, rng, stale, o1, o2);
  T* pk = package_ptr<Mo>(reinterpret_cast<T*>(a.b.state), a.b.n_envs, j, a.c.history, (int)(p & (uint32_t)(kPackSlots - 1)));
#pragma unroll
  for (int q = 0; q < L.n_quads; ++q) store_quad_at(pk, q, &g.w[4 * q]);
#pragma unroll
  for (int q = 0; q < (2 * C + 3) / 4; ++q) {
    T v[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = 4 * q + l;
      v[l] = idx < C ? o1[idx < C ? idx : 0] : idx < 2 * C ? o2[idx < 2 * C && idx >= C ? idx - C : 0] : T(0);
    }
    store_quad_at(pk, L.n_quads + q, v);
  }
}

// Regenerates pending packages of the 32 environments of a warp, one package per lane and pass (called by
// all 32 lanes together; `e_mine` / `pend` are the caller lane's episode index and pending bits, the new
// pending bits are returned).  Work items of a pass: the packages some lane needs NEXT first, then the
// other pending slot-0 packages in lane order, slot 1, ...  One pass; more only if more than 32 lanes
// were waiting for their next package (impossible: one per lane).
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__device__ __forceinline__ int flush_pending(const KArgs<T>& a, int64_t warp_base, uint32_t e_mine, int pend) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int next = (int)((e_mine + 1) & (kPackSlots - 1));
  // group 0: the next-needed slot of each lane where that slot is pending; groups 1..kPackSlots: slot s - 1
  // of each lane where pending and not already in group 0
  unsigned b[kPackSlots + 1];
  int start[kPackSlots + 2];
  b[0] = __ballot_sync(full, (pend >> next) & 1);
  start[0] = 0;
  start[1] = __popc(b[0]);
#pragma unroll
  for (int s = 0; s < kPackSlots; ++s) {
    b[s + 1] = __ballot_sync(full, ((pend >> s) & 1) && s != next);
    start[s + 2] = start[s + 1] + __popc(b[s + 1]);
  }
  const int total = start[kPackSlots + 1];
  int grp = -1, src = 0;
  const bool has = lane < total;
#pragma unroll
  for (int g = 0; g <= kPackSlots; ++g)
    if (has && lane >= start[g] && lane < start[g + 1]) { grp = g; src = (int)__fns(b[g], 0, lane - start[g] + 1); }
  const uint32_t e_src = __shfl_sync(full, e_mine, src);
  if (has) {
    const uint32_t slot = grp == 0 ? ((e_src + 1) & (kPackSlots - 1)) : (uint32_t)(grp - 1);
    // slot s holds a package p > e with p = s (mod kPackSlots): the first one the owner will ask this slot for
    // (modulo 2^28 like e: a multiple of kPackSlots, so the slot of p is unchanged)
    const uint32_t p = (e_src + 1 + ((slot - (e_src + 1)) & (kPackSlots - 1))) & kEpMask;
    gen_package<T, TASK, PHYS, NOISE, RNG, PID>(a, warp_base + src, p);
  }
  // which of my pending packages were among the first 32 items
  if (((pend >> next) & 1) && __popc(b[0] & ((1u << lane) - 1u)) < 32) pend &= ~(1 << next);
#pragma unroll
  for (int s = 0; s < kPackSlots; ++s)
    if (((pend >> s) & 1) && s != next && start[s + 1] + __popc(b[s + 1] & ((1u << lane) - 1u)) < 32) pend &= ~(1 << s);
  __syncwarp();                                            // package stores -> visible to the lanes that load them
  return pend;
}

// A finished environment takes its next package: everything a reset writes comes from the package,
// the words a reset keeps (OU state, gyro bias, episode counters of the pool) stay, and the carried
// words enter the gyro chain of the two reset observations linearly:
//   b1 = pi b0 + s n1            lp1 = (1-r) stale + r (om + b1 + W n1')
//   b2 = pi b1 + s n2            lp2 = (1-r) lp1   + r (om + b2 + W n2')
// (sensors.py:121-134, envs/utils.py:76-79; the package holds the b0 = stale = 0 solution).
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__device__ __forceinline__ void take_package(Model<T, TASK, PHYS, NOISE, RNG, PID>& m, T* state, int64_t n, int64_t i,
                                             int history, const T stale[3], T* o1, T* o2) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  constexpr int C = Mo::C;
  const DevCfg<T>& c = m.c;
  T* w = m.w;
  const uint32_t ew = ep_word(w[L.ep_index]);        // (e << 4) | pending bits
  const int slot = (int)(((ew >> 4) + 1) & (kPackSlots - 1));
  const T* pk = package_ptr<Mo>(state, n, i, history, slot);
  T ou[4], b0[3] = {T(0), T(0), T(0)};
#pragma unroll
  for (int k = 0; k < 4; ++k) ou[k] = w[L.ou + k];
  if constexpr (NOISE) {
#pragma unroll
    for (int k = 0; k < 3; ++k) b0[k] = w[L.gyro_bias + k];
  }
#pragma unroll
  for (int q = 0; q < L.n_quads; ++q) load_quad_at(pk, q, &w[4 * q]);
#pragma unroll
  for (int q = 0; q < (2 * C + 3) / 4; ++q) {
    T v[4];
    load_quad_at(pk, L.n_quads + q, v);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = 4 * q + l;
      if (idx < C) o1[idx < C ? idx : 0] = v[l];
      else if (idx < 2 * C) o2[idx < 2 * C && idx >= C ? idx - C : 0] = v[l];
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) w[L.ou + k] = ou[k];
  if constexpr (NOISE) {
    const T r = c.lpf_ratio, pi1 = c.gyro_pi, pi2 = c.gyro_pi * c.gyro_pi;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const T d1 = (T(1) - r) * stale[k] + r * (pi1 * b0[k]);          // lp1 - lp1'
      const T d2 = (T(1) - r) * d1 + r * (pi2 * b0[k]);                // lp2 - lp2'
      o1[10 + k] += d1;
      o2[10 + k] += d2;
      w[L.gyro_lpf + k] += d2;
      w[L.gyro_bias + k] += pi2 * b0[k];
    }
  }
  set_ep_word(w[L.ep_index], (ew + 16) | (1u << slot));   // (32-bit wrap: e + 1 modulo 2^28)
}

// ---------------------------------------------------------------------------------------------
//  constructor: zero state, nominal parameters, base.py:143's compute_observation()
// ---------------------------------------------------------------------------------------------
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__global__ void __launch_bounds__(kMaxBlock) k_init(const __grid_constant__ KArgs<T> a) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  const int64_t n = a.b.n_envs;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Mo m(a.c);
  const DevCfg<T>& c = a.c;
  init_nominal(m);
  if constexpr (NOISE) {
    const Rng<T, RNG> rng = make_rng<T, RNG>(a, a.counter, i, a.b.tape_init, a.dump_init);
    T z[3];
    rng.template normals<3>(SITE_INIT, 12, z);
#pragma unroll
    for (int k = 0; k < 3; ++k) m.w[L.gyro_bias + k] = c.gyro_sigma_b * z[k];
  }
  T* state = reinterpret_cast<T*>(a.b.state);
  m.store(state, n, i, true);
  const T zero[4] = {T(0), T(0), T(0), T(0)};
  for (int qd = 0; qd < (c.history - 1) * Mo::QH; ++qd) store_quad(state, n, i, L.n_quads + qd, zero);
  if constexpr (RNG == PDX_RNG_PHILOX) {                   // the first two reset packages of every environment
#pragma unroll 1
    for (uint32_t p = 1; p <= (uint32_t)kPackSlots; ++p) gen_package<T, TASK, PHYS, NOISE, RNG, PID>(a, i, p);
  } else {
    for (int qd = 0; qd < kPackSlots * L.pack_quads; ++qd) store_quad(state, n, i, pool_plane<Mo>(c.history) + qd, zero);
  }
}

// ---------------------------------------------------------------------------------------------
//  explicit reset of all / masked environments (dense: one thread per env)
// ---------------------------------------------------------------------------------------------
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
__global__ void __launch_bounds__(kMaxBlock) k_reset(const KArgs<T> a) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  constexpr int C = Mo::C, E = Mo::E, QH = Mo::QH;
  const int64_t n = a.b.n_envs;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (a.mask && !a.mask[i]) return;
  Mo m(a.c);
  T* state = reinterpret_cast<T*>(a.b.state);
  m.load(state, n, i);
  const Rng<T, RNG> rng = make_rng<T, RNG>(a, a.counter, i, a.b.tape_reset, a.dump_reset);
  T stale[3], o1[C], o2[C];
  m.body_rates(stale);
  reset_env(m, rng, stale, o1, o2);
  m.store(state, n, i, true);
  const int H = a.c.history;
  const T* la = &m.w[L.last_action];
  T* row = reinterpret_cast<T*>(a.b.obs) + i * a.c.obs_dim;
  for (int j = 0; j < H; ++j) {
    const bool newest = j == H - 1;
#pragma unroll
    for (int k = 0; k < C; ++k) row[j * E + k] = newest ? o2[k] : o1[k];
#pragma unroll
    for (int k = 0; k < 4; ++k) row[j * E + C + k] = la[k];
  }
  store_history<T, E, QH>(state, n, i, L.n_quads, H, [&](int s, int idx) {
    return idx < C ? (s == H - 2 ? o2[idx < C ? idx : 0] : o1[idx < C ? idx : 0]) : la[idx - C < 4 && idx >= C ? idx - C : 0];
  });
}

// CAS-based min/max on doubles for the episode statistics
__device__ __forceinline__ void atomic_min_double(double* addr, double v) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *p;
  while (__longlong_as_double((long long)old) > v) {
    const unsigned long long assumed = old;
    old = atomicCAS(p, assumed, (unsigned long long)__double_as_longlong(v));
    if (old == assumed) break;
  }
}
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *p;
  while (__longlong_as_double((long long)old) < v) {
    const unsigned long long assumed = old;
    old = atomicCAS(p, assumed, (unsigned long long)__double_as_longlong(v));
    if (old == assumed) break;
  }
}

// Episode statistics of a block -> the 8-word global vector: per-thread columns in shared memory
// (n, sum ret, sum ret^2, sum len; min/max ret, min/max len), one warp-shuffle reduction and one set
// of atomics per block and launch.  Called by ALL threads of the block (it contains a barrier).
template <class T>
__device__ __forceinline__ void block_reduce_episode_stats(double* gs, const double* acc_sum, const T* acc_ext, int B, bool any_fin) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (gs && __syncthreads_or(any_fin ? 1 : 0)) {
    if (warp == 0) {
      double v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = (k == 4 || k == 6) ? 1e300 : (k == 5 || k == 7) ? -1e300 : 0.0;
      for (int col = lane; col < B; col += 32) {
        if (acc_sum[col] > 0.0) {
#pragma unroll
          for (int k = 0; k < 4; ++k) v[k] += acc_sum[k * B + col];
          v[4] = fmin(v[4], (double)acc_ext[0 * B + col]); v[5] = fmax(v[5], (double)acc_ext[1 * B + col]);
          v[6] = fmin(v[6], (double)acc_ext[2 * B + col]); v[7] = fmax(v[7], (double)acc_ext[3 * B + col]);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        v[4] = fmin(v[4], __shfl_xor_sync(0xffffffffu, v[4], o));
        v[5] = fmax(v[5], __shfl_xor_sync(0xffffffffu, v[5], o));
        v[6] = fmin(v[6], __shfl_xor_sync(0xffffffffu, v[6], o));
        v[7] = fmax(v[7], __shfl_xor_sync(0xffffffffu, v[7], o));
      }
      if (lane == 0) {
        atomicAdd(&gs[0], v[0]); atomicAdd(&gs[1], v[1]); atomicAdd(&gs[2], v[2]); atomicAdd(&gs[3], v[3]);
        atomic_min_double(&gs[4], v[4]); atomic_max_double(&gs[5], v[5]);
        atomic_min_double(&gs[6], v[6]); atomic_max_double(&gs[7], v[7]);
      }
    }
  }
}

// OR of `pred` over the `n_threads` threads (a multiple of 32) that meet at named barrier `bar_id` (1..15; 0 is
// __syncthreads): the package vote of a 128-thread group in k_rollout and of a tile in k_collect
__device__ __forceinline__ bool tile_vote(int bar_id, int n_threads, bool pred) {
  uint32_t out;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %3, 0;\n\t"
      "barrier.cta.red.or.pred q, %1, %2, p;\n\t"
      "selp.u32 %0, 1, 0, q;\n\t}\n"
      : "=r"(out)
      : "r"(bar_id), "r"(n_threads), "r"((uint32_t)pred)
      : "memory");
  return out != 0;
}

// ---- bulk asynchronous copy shared -> global (TMA engine), bulk-group completion ------------
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Shared-memory plan of k_rollout (dynamic shared memory), B threads = W warps:
//   T tile0, tile1 [B][D]        observation rows; warp w owns rows [32 w, 32 w + 32) of each tile, which
//                                have exactly the layout of its slice of the row-major [n_envs][D]
//                                output (tile1 only when n_tiles == 2)
//   T stage [W][E][32]           only when D is a multiple of 16: column-major staging of the new entry
//   T acc_ext [4][B], double acc_sum [4][B]   per-thread episode statistics (min/max ret, min/max len;
//                                n, sum ret, sum ret^2, sum len), reduced once per launch
//   Row modes (template parameter WIDE of the kernel):
//     0  rows as in the output, walked word by word                (D not a multiple of 16)
//     1  same layout, every lane walks its row rotated by its lane id, the new entry goes through `stage`
//     2  rows padded by 16 bytes (an odd number of 16-byte vectors per row: 128-bit accesses of a quarter warp fall
//        into eight different bank groups), history shifted with 128-bit loads / stores, every lane sends its own
//        row with one bulk copy.  float32 rows whose entries are whole 16-byte vectors (Circle, TakeOff), long
//        histories: D = 160 ran 75 % bank-conflict wavefronts in mode 1 (profiles/r2_h8.summary.csv)
__host__ __device__ inline int rollout_row_stride(int D, int wmode, size_t elem) { return wmode == 2 ? D + (int)(16 / elem) : D; }
template <class T>
__host__ __device__ inline size_t rollout_smem_bytes(int block, int D, int n_tiles, int E, int wmode) {
  size_t words = (size_t)n_tiles * block * rollout_row_stride(D, wmode, sizeof(T)) + (size_t)4 * block;
  if (wmode == 1) words += (size_t)(block / 32) * E * 32;
  size_t bytes = (words * sizeof(T) + 15) & ~(size_t)15;
  return bytes + sizeof(double) * 4 * block;
}

// N consecutive float words of a thread's shared-memory row written as 64-bit stores: `dst` 8-byte aligned (ALIGNED)
// or 4 bytes past an 8-byte boundary (one scalar store first).  fast2 rows are 2 E words long, so a row starts 8-byte
// aligned and its second entry does when E is even.  Halves the store instructions of the row writes, and a
// half warp's 64-bit accesses at the 34-word row stride are bank-conflict free (the 32-bit ones are 2-way).
template <int N, bool ALIGNED>
__device__ __forceinline__ void store_words64(float* dst, const float (&v)[N]) {
  constexpr int first = ALIGNED ? 0 : 1;
  if (!ALIGNED) dst[0] = v[0];
#pragma unroll
  for (int k = first; k + 1 < N; k += 2) *reinterpret_cast<float2*>(dst + k) = make_float2(v[k], v[k + 1]);
  if ((N - first) & 1) dst[N - 1] = v[N - 1];
}

// per-thread context of the step loop: everything that is not the environment state itself
template <class T>
struct StepCtx {
  T* state;
  int64_t n, i;               // environments of the shard, this thread's (local) environment index
  bool valid;                 // i < n
  int lane, tid, B;           // lane in the warp, thread in the block, threads per block (statistics columns)
  T* row0; T* row1;           // this thread's row in the two observation tiles (row1 == row0 with one tile)
  T* stg;                     // column-major staging buffer of the warp (WIDE == 1 only)
  int RS;                     // words between the rows of two neighbouring lanes in a tile
  double* acc_sum; T* acc_ext;
  int NT;                     // observation tiles (1 or 2)
  bool fast2, bulk, latency, any_fin;
  T ev_reward, ev_cost;       // EVAL: this step's reward, cost and flags, handed to the caller
  bool ev_terminated, ev_truncated;
};

// ---------------------------------------------------------------------------------------------
//  ONE env.step (+ auto-reset) of every environment of the calling thread group, with the state in the
//  registers of `m`: shared by k_rollout (open-loop action sequences) and k_collect (csrc/pdx_collect.cu:
//  the policy step runs between two calls).  `a4`: this thread's action; outputs of step t go to row t of the
//  time-major buffers in a.b.  `vote(pred)`: OR of `pred` over the thread group that regenerates reset
//  packages together (a barrier: all threads of the group call it once per step).
// ---------------------------------------------------------------------------------------------
// WIDE: row mode (see rollout_smem_bytes) -- a template parameter because as a run-time branch it made ptxas spill
// the 17 words of the new entry on BOTH paths.
// EVAL (k_evaluate, csrc/pdx_evaluate.cu): no global per-step stores (observation rows and their bulk copies, reward,
// cost, flags, episode return / length, final_obs) and no episode statistics; reward, cost and flags go to sc.ev_*.
// Without auto-reset (an evaluation) no reset package is ever taken, so the package regeneration and its vote are
// compiled out as well: `vote` is not called.
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID, int WIDE, bool EVAL = false, class Vote>
__device__ __forceinline__ void rollout_step(const KArgs<T>& a, Model<T, TASK, PHYS, NOISE, RNG, PID>& m, StepCtx<T>& sc,
                                             const int t, const float4 a4, Vote vote) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  constexpr int C = Mo::C, E = Mo::E;
  constexpr bool POOL = RNG == PDX_RNG_PHILOX;       // pre-computed reset packages (see gen_package)
  constexpr bool quad = WIDE == 2 && sizeof(T) == 4 && E % 4 == 0 && C % 4 == 0;
  constexpr bool wide = WIDE == 1 || (WIDE == 2 && !quad);
  const DevCfg<T>& c = a.c;
  const int64_t n = sc.n, i = sc.i;
  const bool valid = sc.valid, fast2 = sc.fast2, bulk = sc.bulk, latency = sc.latency;
  const int lane = sc.lane, tid = sc.tid, B = sc.B, NT = sc.NT;
  const int D = c.obs_dim, H = c.history;
  const unsigned full = 0xffffffffu;
  T* state = sc.state;
  T* stg = sc.stg;
  double* acc_sum = sc.acc_sum;
  T* acc_ext = sc.acc_ext;
  T* w = m.w;
  T* tn = (t & 1) ? sc.row1 : sc.row0;               // this step's row, previous step's row
  const T* to = (t & 1) ? sc.row0 : sc.row1;
  const int64_t tn_off = (int64_t)t * n;             // offset of step t in the [n_steps][n] outputs
  bool fin = false, dn = false, trunc = false, state_ok = true;
  T ep_ret_out = T(0);
  int ep_len_out = 0;
  T core[C], a_new[4], actT[4];
  const int n_ep = (int)w[L.ep_length] + 1;          // 1-based step index in the episode
  const float act[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) actT[k] = (T)act[k];

    // ---- this step's tile slice was last read by the warp's bulk copy of step t - n_tiles (lane 0 issues
    // the copies of the warp, so it is the lane that can wait for them).  No block-wide barrier: warps
    // run through their steps independently.
    if (!EVAL && !fast2) {
      if (lane == 0 || quad) { if (NT == 2) bulk_wait_read<1>(); else bulk_wait_read<0>(); }   // (quad: a lane sends its own row)
      __syncwarp();
    }

    // ---- history part of the row first (it does not depend on this step's arithmetic):
    // [o(k-H+1), a(k-H), ..., o(k-1), a(k-2)] = entries 1..H-1 of the previous row (base.py:303-319).
    // The tile has the row-major layout of the output, so lane l's row starts at bank l*D mod 32: when D is
    // a multiple of 16 a warp walking its rows in step hits few banks (D = 160: ONE bank).  Each lane
    // then walks its row rotated by its lane id (bank l*(D+1) + k: conflict free).
    // quirk (Bullet agent): after a reset the action deque holds H references to ring[-1]
    // (agents.py:386, base.py:426-427), which the latency ring overwrites in place with the current action
    // -> those entries read as the *current* action for as long as they stay in the deque.
    if (valid) {
      if constexpr (quad) {
        constexpr int VPE = E / 4;                         // 16-byte vectors per entry; the action is the last one
        const float4* src = reinterpret_cast<const float4*>(to) + VPE;
        float4* dst = reinterpret_cast<float4*>(tn);
        for (int j = 0; j < H - 1; ++j) {
          const bool alias = latency && (j + n_ep <= H);
#pragma unroll
          for (int q = 0; q < VPE; ++q) {
            float4 v = src[j * VPE + q];
            if (q == VPE - 1 && alias) v = make_float4((float)actT[0], (float)actT[1], (float)actT[2], (float)actT[3]);
            dst[j * VPE + q] = v;
          }
        }
      } else if constexpr (wide) {
        for (int j = 0; j < H - 1; ++j) {
          const bool alias = latency && (j + n_ep <= H);
#pragma unroll
          for (int k = 0; k < E; ++k) {
            int kk = k + lane;
            kk = kk >= E ? kk - E : kk;
            kk = kk >= E ? kk - E : kk;
            T v = to[(j + 1) * E + kk];
            if (alias && kk >= C) v = kk == C ? actT[0] : kk == C + 1 ? actT[1] : kk == C + 2 ? actT[2] : actT[3];
            tn[j * E + kk] = v;
          }
        }
      } else if (fast2) {                                  // entry 0 is already there; only the aliasing quirk
        if (latency && n_ep <= H) {
#pragma unroll
          for (int k = 0; k < 4; ++k) tn[C + k] = actT[k];
        }
      } else {
        for (int j = 0; j < H - 1; ++j) {
          const bool alias = latency && (j + n_ep <= H);
#pragma unroll
          for (int k = 0; k < E; ++k) {
            T v = to[(j + 1) * E + k];
            if (k >= C && alias) v = actT[k >= C ? k - C : 0];
            tn[j * E + k] = v;
          }
        }
      }
    }

    if (valid) {
      const Rng<T, RNG> rng = make_rng<T, RNG>(a, a.counter + (uint64_t)t, i,
                                               a.b.tape_step ? a.b.tape_step + (int64_t)t * c.slots_step * n : nullptr,
                                               a.dump_step ? a.dump_step + (int64_t)t * c.slots_step * n : nullptr);
      T la_prev[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) la_prev[k] = w[L.last_action + k];

      // ---- physics sub-steps; the observation call after each one is discarded by the
      // reference (base.py:464) but advances the gyro bias / low-pass state (quirk A.6-1)
      int slot = 0;
      for (int s = 0; s < c.agg; ++s) {
        const bool full_obs = (s % c.obs_rate) == 0;
        m.substep(rng, act, s, slot, full_obs);
        slot += 4 + (NOISE ? (full_obs ? c.slots_obs_full : c.slots_obs_gyro) : 0);
      }

      T target[3] = {c.target[0], c.target[1], c.target[2]};
      if constexpr (TASK == PDX_TASK_CIRCLE) m.ref_point((n_ep + (int)w[L.ref_offset]) % 300, target);   // circle.py:130
      if constexpr (TASK == PDX_TASK_TAKEOFF) m.ref_point(min(n_ep * c.agg, 299), target);                // takeoff.py:108

      // ---- does the episode end with this step?  Known as soon as the physics is done (compute_done,
      // TimeLimit of __init__.py:11): a lane that will take a reset package at the end of the step asks
      // for its cache lines NOW, a thousand instructions before it reads them.
      {
        T e[3], om[3];
        m.euler(e);
        m.body_rates(om);
        dn = m.done(e, om, target);
        trunc = n_ep >= c.max_episode_steps;
        if (c.reset_on_nonfinite) {
          // extension: a non-finite state ends the episode as a truncation that carries no reward and no cost
          // (the collector bootstraps a truncation with V(final observation), which is sanitised below)
#pragma unroll
          for (int k = 0; k < 6; ++k) state_ok = state_ok && M<T>::finite(w[L.xyz + k]);
#pragma unroll
          for (int k = 0; k < 3; ++k) state_ok = state_ok && M<T>::finite(om[k]) && M<T>::finite(e[k]);
          trunc = trunc || !state_ok;
        }
        fin = dn || trunc;
        if constexpr (POOL) {
          if (fin && c.auto_reset) {
            const char* pk = reinterpret_cast<const char*>(
                package_ptr<Mo>(state, n, i, H, (int)(((ep_word(w[L.ep_index]) >> 4) + 1) & (kPackSlots - 1))));
#pragma unroll
            for (int b = 0; b < (int)(L.pack_quads * 4 * sizeof(T)) + 127; b += 128)
              asm volatile("prefetch.global.L1 [%0];" ::"l"(pk + b));     // (into L1: this lane reads them itself)
          }
        }
      }

      // ---- the observation that is returned (base.py:468 -> compute_history)
      T q_true[4] = {T(0), T(0), T(0), T(1)};
      if constexpr (!NOISE) {
        if constexpr (Mo::BULLET) { for (int k = 0; k < 4; ++k) q_true[k] = w[L.quat + k]; }
        else quat_from_euler(w[L.rpy], w[L.rpy + 1], w[L.rpy + 2], q_true);
      }
      m.observe(rng, SITE_FINAL_OBS, slot, target, actT, q_true, core);

      // a(k-1) paired with o(k); Bullet aliasing quirk as above
      {
        const bool alias = latency && (H - 1 + n_ep <= H);
#pragma unroll
        for (int k = 0; k < 4; ++k) a_new[k] = alias ? actT[k] : la_prev[k];
      }
    }

    // ---- newest entry of the row: [o(k), a(k-1)]
    if constexpr (quad) {
      if (valid) {
        float4* dst = reinterpret_cast<float4*>(tn + (H - 1) * E);
#pragma unroll
        for (int q = 0; q < C / 4; ++q)
          dst[q] = make_float4((float)core[4 * q], (float)core[4 * q + 1], (float)core[4 * q + 2], (float)core[4 * q + 3]);
        dst[C / 4] = make_float4((float)a_new[0], (float)a_new[1], (float)a_new[2], (float)a_new[3]);
      }
    } else if constexpr (wide) {                           // registers cannot be indexed by the rotated position:
#pragma unroll                                             // column-major staging buffer of the warp
      for (int k = 0; k < C; ++k) stg[k * 32 + lane] = core[k];
#pragma unroll
      for (int k = 0; k < 4; ++k) stg[(C + k) * 32 + lane] = a_new[k];
      __syncwarp();
      if (valid) {
#pragma unroll
        for (int k = 0; k < E; ++k) {
          int kk = k + lane;
          kk = kk >= E ? kk - E : kk;
          kk = kk >= E ? kk - E : kk;
          tn[(H - 1) * E + kk] = stg[kk * 32 + lane];
        }
      }
      __syncwarp();
    } else {                                               // other strides: at most 8-way (measured faster)
      if (fast2) {                                         // the other tile: its bulk copy (issued a step ago) must have
        if (lane == 0) bulk_wait_read<0>();                // been read out before entry 0 of the next row goes in
        __syncwarp();
      }
      if (valid) {
        if constexpr (sizeof(T) == 4) {
          if (fast2) {                                     // H == 2: entry 1 of this row, entry 0 of the next one
            float ent[E];
#pragma unroll
            for (int k = 0; k < C; ++k) ent[k] = (float)core[k];
#pragma unroll
            for (int k = 0; k < 4; ++k) ent[C + k] = (float)a_new[k];
            store_words64<E, (E & 1) == 0>(reinterpret_cast<float*>(tn) + E, ent);
            store_words64<E, true>(reinterpret_cast<float*>(const_cast<T*>(to)), ent);
          }
        }
        if (!(sizeof(T) == 4 && fast2)) {
#pragma unroll
          for (int k = 0; k < C; ++k) tn[(H - 1) * E + k] = core[k];
#pragma unroll
          for (int k = 0; k < 4; ++k) tn[(H - 1) * E + C + k] = a_new[k];
          if (fast2) {
            T* nx = const_cast<T*>(to);
#pragma unroll
            for (int k = 0; k < C; ++k) nx[k] = core[k];
#pragma unroll
            for (int k = 0; k < 4; ++k) nx[C + k] = a_new[k];
          }
        }
      }
    }

    if (valid) {
      // ---- reward / cost / done
      T target[3] = {c.target[0], c.target[1], c.target[2]};
      if constexpr (TASK == PDX_TASK_CIRCLE) m.ref_point((n_ep + (int)w[L.ref_offset]) % 300, target);
      if constexpr (TASK == PDX_TASK_TAKEOFF) m.ref_point(min(n_ep * c.agg, 299), target);
      T e[3], om[3];
      m.euler(e);
      m.body_rates(om);
      // action penalties are float32 arithmetic in the reference (float32 action array)
      float nca2 = 0.0f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float v = 0.5f * (fminf(fmaxf(act[k], -1.0f), 1.0f) + 1.0f);
        nca2 += v * v;
      }
      const T pa = (T)((float)c.pen_action * sqrtf(nca2));
      T par = T(0);
      if constexpr (TASK == PDX_TASK_CIRCLE) {                        // circle.py:186 (hover/takeoff: == 0, A.6-10)
        T d2 = T(0);
        if (!(latency && n_ep == 1)) {
#pragma unroll
          for (int k = 0; k < 4; ++k) { const T d = actT[k] - w[L.last_action + k]; d2 += d * d; }
        }
        par = c.arp * M<T>::sqrt(d2);
      }
      const T prpy = c.pen_angle * norm3(e[0], e[1], e[2]);
      const T pspin = c.pen_spin * norm3(om[0], om[1], om[2]);
      const T pterm = dn ? c.pen_terminal : T(0);
      const T cvel = TASK == PDX_TASK_TAKEOFF ? c.pen_action : c.pen_velocity;   // takeoff.py:165
      const T pvel = cvel * norm3(w[L.vel], w[L.vel + 1], w[L.vel + 2]);
      const T penalties = ((((prpy + par) + pspin) + pvel) + pa) + pterm;
      const T dist = norm3(w[L.xyz] - target[0], w[L.xyz + 1] - target[1], w[L.xyz + 2] - target[2]);
      T r = -dist - penalties;
      if (TASK == PDX_TASK_TAKEOFF && w[L.xyz + 2] < T(0.08)) r -= T(1);
      T cst = m.cost(e, om, act);

      // ---- episode accounting
      if (c.reset_on_nonfinite && !state_ok) { r = T(0); cst = T(0); }
      w[L.ep_return] += r;
      w[L.ep_length] = (T)n_ep;
#pragma unroll
      for (int k = 0; k < 4; ++k) w[L.last_action + k] = actT[k];
      if constexpr (EVAL) {
        sc.ev_reward = r; sc.ev_cost = cst; sc.ev_terminated = dn; sc.ev_truncated = trunc;
      } else {
        reinterpret_cast<T*>(a.b.reward)[tn_off + i] = r;
        reinterpret_cast<T*>(a.b.cost)[tn_off + i] = cst;
        a.b.terminated[tn_off + i] = dn ? 1 : 0;
        a.b.truncated[tn_off + i] = trunc ? 1 : 0;
        ep_ret_out = w[L.ep_return];
        ep_len_out = n_ep;
        if (a.b.episode_return) reinterpret_cast<T*>(a.b.episode_return)[tn_off + i] = fin ? ep_ret_out : T(0);
        if (a.b.episode_length) a.b.episode_length[tn_off + i] = fin ? ep_len_out : 0;
      }
    }
    if constexpr (EVAL) return;

    // ---- finished episodes: statistics, auto-reset
    if (fin) {
      sc.any_fin = true;
      acc_sum[0 * B + tid] += 1.0;
      acc_sum[1 * B + tid] += (double)ep_ret_out;
      acc_sum[2 * B + tid] += (double)ep_ret_out * (double)ep_ret_out;
      acc_sum[3 * B + tid] += (double)ep_len_out;
      acc_ext[0 * B + tid] = M<T>::fmin(acc_ext[0 * B + tid], ep_ret_out);
      acc_ext[1 * B + tid] = M<T>::fmax(acc_ext[1 * B + tid], ep_ret_out);
      acc_ext[2 * B + tid] = M<T>::fmin(acc_ext[2 * B + tid], (T)ep_len_out);
      acc_ext[3 * B + tid] = M<T>::fmax(acc_ext[3 * B + tid], (T)ep_len_out);
    }
    const bool do_reset = fin && c.auto_reset;
    const unsigned ballot = __ballot_sync(full, do_reset);
    if (ballot) {
      if (do_reset && a.b.final_obs) {                     // last observation of the episode
        T* fo = reinterpret_cast<T*>(a.b.final_obs) + (tn_off + i) * D;
        if (c.reset_on_nonfinite) { for (int k = 0; k < D; ++k) fo[k] = M<T>::finite(tn[k]) ? tn[k] : T(0); }
        else { for (int k = 0; k < D; ++k) fo[k] = tn[k]; }
      }
      if (do_reset) {
        T o1[C], o2[C], stale[3];
        m.body_rates(stale);
        if (c.reset_on_nonfinite) {                        // extension: do not seed the next episode's
#pragma unroll
          for (int k = 0; k < 3; ++k) if (!M<T>::finite(stale[k])) stale[k] = T(0);   // low pass with inf / NaN
        }
        if constexpr (POOL) {
          take_package(m, state, n, i, H, stale, o1, o2);
        } else {
          // the draws of auto-reset number e + 1 of this environment (same keys as gen_package in dump mode)
          const uint32_t e_next = ((ep_word(w[L.ep_index]) >> 4) + 1) & kEpMask;
          const Rng<T, RNG> rr = make_rng<T, RNG>(a, (uint64_t)e_next, i,
                                                  a.b.tape_reset ? a.b.tape_reset + (int64_t)t * c.slots_reset * n : nullptr,
                                                  a.dump_reset ? a.dump_reset + (int64_t)t * c.slots_reset * n : nullptr, true);
          reset_env(m, rr, stale, o1, o2);
          set_ep_word(w[L.ep_index], e_next << 4);
        }
        bool rows_done = false;
        if constexpr (sizeof(T) == 4) {
          if (fast2) {                                     // H == 2: the whole row [o1 a | o2 a] and entry 0 of the next
            float rw[2 * E];
#pragma unroll
            for (int k = 0; k < C; ++k) { rw[k] = (float)o1[k]; rw[E + k] = (float)o2[k]; }
#pragma unroll
            for (int k = 0; k < 4; ++k) { rw[C + k] = (float)w[L.last_action + k]; rw[E + C + k] = (float)w[L.last_action + k]; }
            store_words64<2 * E, true>(reinterpret_cast<float*>(tn), rw);
            float ent[E];
#pragma unroll
            for (int k = 0; k < E; ++k) ent[k] = rw[E + k];
            store_words64<E, true>(reinterpret_cast<float*>(const_cast<T*>(to)), ent);
            rows_done = true;
          }
        }
        if (!rows_done) {
          for (int j = 0; j < H; ++j) {                    // first observation of the new episode
#pragma unroll
            for (int k = 0; k < C; ++k) tn[j * E + k] = (j == H - 1) ? o2[k] : o1[k];
#pragma unroll
            for (int k = 0; k < 4; ++k) tn[j * E + C + k] = w[L.last_action + k];
          }
          if (fast2) {
            T* nx = const_cast<T*>(to);
#pragma unroll
            for (int k = 0; k < C; ++k) nx[k] = o2[k];
#pragma unroll
            for (int k = 0; k < 4; ++k) nx[C + k] = w[L.last_action + k];
          }
        }
      }
    }
    if constexpr (POOL) {
      // Package regeneration is decided per vote group (`vote`: a 128-thread group of k_rollout's block, a tile
      // of k_collect), one barrier vote per step: all warps of a group run the
      // (long) generator at the same step, and the barrier keeps them within one step of each other -- the
      // step loop is ~30 KB of straight-line code, and warps that drift apart each stream it through the
      // instruction caches on their own (measured: `no_instruction` became the top stall).  The vote
      // passes when a warp has a good pass worth of packages pending (40: every lane of the pass busy), or
      // when some environment would find its NEXT slot still pending (all kPackSlots of its packages
      // used up since the last regeneration: a burst of very short episodes) -- so the take at the end of
      // a step never has to wait for a package.
      const uint32_t ew = ep_word(w[L.ep_index]), e0 = ew >> 4;
      const int pend0 = (int)(ew & 15);
      const int total = (int)__reduce_add_sync(full, (unsigned)__popc(pend0));     // pending packages of the warp
      const bool urgent = (pend0 >> ((e0 + 1) & (kPackSlots - 1))) & 1;
      if (vote(urgent || total >= 40)) {
        if (valid) m.store(state, n, i, true);             // the state is parked in its own planes around the
        // generator: nothing is live across it (inlined on top of the live state it spilled on the hot path)
        const int pend1 = flush_pending<T, TASK, PHYS, NOISE, RNG, PID>(a, i - lane, e0, pend0);
        if (valid) m.load(state, n, i);
        else {
#pragma unroll
          for (int k = 0; k < Mo::NW; ++k) w[k] = T(0);
        }
        set_ep_word(w[L.ep_index], (ew & ~15u) | (uint32_t)pend1);
      }
    }

    // ---- the warp's rows of this step leave as one bulk copy (or a flat coalesced copy when the
    // destination does not meet the 16-byte rules of the bulk engine)
    const int64_t warp_base = i - lane;                  // first environment of this warp
    const int rows_w = (int)max((int64_t)0, min((int64_t)32, n - warp_base));     // rows of this warp's tile slice
    if (rows_w > 0) {
      T* gdst = reinterpret_cast<T*>(a.b.obs) + (tn_off + warp_base) * D;
      const T* wt = tn - lane * sc.RS;                   // this warp's slice of this step's tile
      if (bulk) {
        fence_async_smem();
        if constexpr (quad) {                            // padded rows: one copy per row, issued by its lane
          if (valid) bulk_store(gdst + lane * D, tn, (uint32_t)D * (uint32_t)sizeof(T));
        } else {
          __syncwarp();
          if (lane == 0) bulk_store(gdst, wt, (uint32_t)rows_w * (uint32_t)D * (uint32_t)sizeof(T));
        }
      } else {
        __syncwarp();
        if constexpr (quad) {
          for (int r = 0; r < rows_w; ++r)
            for (int k = lane; k < D; k += 32) gdst[r * D + k] = wt[r * sc.RS + k];
        } else {
          for (int e = lane; e < rows_w * D; e += 32) gdst[e] = wt[e];
        }
        __syncwarp();
      }
    }
}

// ---------------------------------------------------------------------------------------------
//  fused multi-step env.step (+ auto-reset)
// ---------------------------------------------------------------------------------------------
template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID, int WIDE>
__global__ void __maxnreg__(128) k_rollout(const __grid_constant__ KArgs<T> a) {
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr Layout L = Mo::L;
  constexpr int E = Mo::E, QH = Mo::QH;
  const DevCfg<T>& c = a.c;
  const int64_t n = a.b.n_envs;
  const int B = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t block_base = (int64_t)blockIdx.x * B;
  const int64_t i = block_base + tid;
  const bool valid = i < n;
  const int D = c.obs_dim, H = c.history;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* tile0 = reinterpret_cast<T*>(smem_raw);
  const int NT = a.n_tiles;
  constexpr bool quad = WIDE == 2 && sizeof(T) == 4 && E % 4 == 0 && Mo::C % 4 == 0;
  constexpr bool wide = WIDE == 1 || (WIDE == 2 && !quad);
  const int RS = rollout_row_stride(D, quad ? 2 : 0, sizeof(T));
  T* tile1 = NT == 2 ? tile0 + (size_t)B * RS : tile0;
  T* stg = tile0 + (size_t)NT * B * RS + (size_t)warp * (E * 32);         // valid only when `wide`
  const size_t words_before_acc = (size_t)NT * B * RS + (wide ? (size_t)(B >> 5) * E * 32 : 0);
  T* acc_ext = tile0 + words_before_acc;
  const size_t off = ((words_before_acc + (size_t)4 * B) * sizeof(T) + 15) & ~(size_t)15;
  double* acc_sum = reinterpret_cast<double*>(smem_raw + off);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    acc_sum[k * B + tid] = 0.0;
    acc_ext[k * B + tid] = (k & 1) ? T(-1e30) : T(1e30);
  }

  Mo m(c);
#pragma unroll
  for (int k = 0; k < Mo::NW; ++k) m.w[k] = T(0);        // lanes past n_envs: no pending packages, never finish
  T* state = reinterpret_cast<T*>(a.b.state);
  T* my_row0 = tile0 + (size_t)tid * RS;
  T* my_row1 = tile1 + (size_t)tid * RS;
  // Programmatic dependent launch: this grid may have started while the kernel before it on the stream is
  // still draining.  Nothing that kernel could have written is touched before griddepcontrol.wait (which
  // returns once it has completed and its writes are visible).  With PDX_BUF_STATE_STABLE the caller
  // guarantees that kernel does not write `state` (collector: it is the policy kernel), so the state
  // load below runs under its tail and only the actions wait.
  const bool state_stable = (a.b.flags & PDX_BUF_STATE_STABLE) != 0;
  if (!state_stable) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }
  // H = 2 with two tiles (the common case): the newest entry of a row is also the oldest entry of the NEXT
  // row, so every entry is written twice -- into this step's tile and into the next step's -- instead of
  // being read back and shifted (17 LDS + their latency at the head of every step).  Not in row mode 2: its
  // history moves with 128-bit copies from the previous row, which the first step reads from tile1.
  const bool fast2 = !wide && !quad && H == 2 && NT == 2;
  if (valid) {
    m.load(state, n, i);
    // history slots -> entries 1..H-1 of the "previous row" (tile1 plays the old tile at t = 0);
    // fast2: straight into entry 0 of the first row
    for (int s = 0; s < H - 1; ++s) {
#pragma unroll
      for (int qd = 0; qd < QH; ++qd) {
        T v[4];
        load_quad(state, n, i, L.n_quads + s * QH + qd, v);
#pragma unroll
        for (int l = 0; l < 4; ++l)
          if (qd * 4 + l < E) { if (fast2) my_row0[qd * 4 + l] = v[l]; else my_row1[(s + 1) * E + qd * 4 + l] = v[l]; }
      }
    }
  }
  if (state_stable) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }
  StepCtx<T> sc;
  sc.state = state; sc.n = n; sc.i = i; sc.valid = valid; sc.lane = lane; sc.tid = tid; sc.B = B;
  sc.row0 = my_row0; sc.row1 = my_row1; sc.stg = stg; sc.RS = RS; sc.acc_sum = acc_sum; sc.acc_ext = acc_ext; sc.NT = NT;
  sc.fast2 = fast2; sc.latency = Mo::BULLET && c.use_latency; sc.any_fin = false;
  // observation rows leave as one bulk copy per warp and step when the destination meets the 16-byte
  // rules of the bulk engine for every step (else: flat coalesced copy by the warp)
  sc.bulk = ((reinterpret_cast<uintptr_t>(a.b.obs) | (uintptr_t)((uint64_t)n * D * sizeof(T))) & 15u) == 0 &&
            (((uint64_t)max((int64_t)0, min((int64_t)32, n - (i - lane))) * D * sizeof(T)) & 15u) == 0;
  const int vote_bar = 1 + (tid >> 7), vote_threads = min(128, B - (tid & ~127));

  for (int t = 0; t < a.n_steps; ++t) {
    // this step's action; the line of step t+1's action is requested now (prefetch: no register is held
    // across the step), so that an L2/HBM miss does not sit at the head of the next step's dependency chain.
    // Into L2: L1 prefetches and a register preload measured no faster, no prefetch 2 % slower (DESIGN.md §4)
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      const float4* ap = reinterpret_cast<const float4*>(a.actions) + (int64_t)t * n + i;
      a4 = *ap;
      if (t + 1 < a.n_steps) asm volatile("prefetch.global.L2 [%0];" ::"l"(ap + n));
    }
    // Package regeneration is voted per 128-thread group of the block (named barrier 1 + group; the last group
    // may be partial): all warps of a group run the (long) generator at the same step, and the barrier keeps
    // them within one step of each other -- the step is ~30 KB of straight-line code, and warps that drift
    // apart each stream it through the instruction caches on their own (measured: `no_instruction` became the
    // top stall).  Barrier 0 belongs to the epilogue's statistics.
    rollout_step<T, TASK, PHYS, NOISE, RNG, PID, WIDE>(a, m, sc, t, a4,
                                                       [&](bool p) { return tile_vote(vote_bar, vote_threads, p); });
  }

  // ---- epilogue: state and history back to HBM, statistics, drain the bulk engine
  if (lane == 0 || quad) bulk_wait_read<0>();
  __syncwarp();
  if (valid) {
    m.store(state, n, i, true);
    const T* last = ((a.n_steps - 1) & 1) ? my_row1 : my_row0;
    store_history<T, E, QH>(state, n, i, L.n_quads, H, [&](int s, int idx) { return last[(s + 1) * E + idx]; });
  }
  block_reduce_episode_stats(a.b.episode_stats, acc_sum, acc_ext, B, sc.any_fin);
  if (lane == 0 || quad) bulk_wait_all();
}

}  // namespace pdx
