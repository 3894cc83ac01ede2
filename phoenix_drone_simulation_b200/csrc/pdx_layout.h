// State layout of one environment, shared by the kernels (compile time) and the C-ABI
// query functions (run time).  Words are `real`s; word w lives in quad w/4, lane w%4 and
// quad q of env i sits at state[(q*n_envs + i)*4 + lane] (one 128-bit access per quad).
//
// The inventory follows SURVEY.md A.8 (what the reference carries between steps):
//   envs/agents.py:52-56 (xyz, xyz_dot, rpy/quaternion, rpy_dot), base.py:261-277 (DR
//   parameters), agents.py:182-186,199-204 (ring, x, A/B/K), envs/utils.py:98 (OU state),
//   sensors.py:68 (gyro bias), envs/utils.py:71 (gyro LPF), base.py:136-137 (history).
#pragma once
#include "../../include/phoenix_b200.h"

namespace pdx {

constexpr int kPackSlots = 4;      // reset packages kept per environment (power of two: slot = package number & 3)
constexpr uint32_t kEpMask = (1u << 28) - 1;   // the auto-reset counter e of the ep_index word counts modulo 2^28

struct Layout {
  int xyz, vel;
  int rpy, omega;          // Simple: Euler angles and body rates are the integrated state
  int quat, omega_world;   // Bullet: quaternion and world angular velocity
  int dt, mass, inertia, ftf1;
  int motor_b, motor_k, motor_x, ring, ring_idx;   // Bullet agent only
  int ou, last_action;
  int pid;                 // PID control modes: rate integral 3, rate last error 3, attitude integral 3,
                           // attitude last error 3 (control.py:133-134,226-227)
  int ep_return, ep_length;
  int ep_index;            // uint32_t (e << 4) | pend: e = number of in-kernel auto-resets this environment
                           // has consumed, modulo 2^28 (keys the reset draws), pend bit s = package slot s was
                           // consumed and is not regenerated yet (one word: the step kernel has no register to
                           // spare).  float64 holds the integer's value, float32 its bit pattern (which may read
                           // as a denormal or a NaN: the word is only moved, never used in arithmetic); see
                           // ep_word / set_ep_word in pdx_kernels.cuh
  int ref_offset;          // circle only
  int gyro_bias, gyro_lpf; // noise only
  int n_words;             // words before the history ring
  int n_dyn_words;         // words that a non-resetting step writes back
  int n_store_quads;       // quads that hold at least one per-step word
  int n_quads;             // ceil(n_words / 4)
  int hist_quads;          // quads per history slot: ceil((C + 4) / 4).  The H-1 slots follow the
                           // n_quads state quads; slot s holds entry s+1 of the last emitted
                           // observation row (= entry s of the next one), base.py:303-319
  int core_dim;            // C
  int pack_quads;          // quads of one pre-computed reset package: the n_quads state quads of a freshly
                           // reset environment followed by the two reset observations (2 C words).  Two
                           // package slots per environment follow the history slots (see k_rollout)
};

constexpr int core_dim_of(int task, bool noise) {
  // hover.py:159-162 (13 / 17 = get_state()), circle.py:169-176 (16), takeoff.py:143-148 (20)
  return task == PDX_TASK_HOVER ? (noise ? 13 : 17) : task == PDX_TASK_CIRCLE ? 16 : 20;
}

constexpr Layout make_layout(int task, int physics, bool noise, bool pid = false) {
  Layout L{};
  int w = 0;
  auto take = [&w](int n) { int o = w; w += n; return o; };
  // ---- words that change every step (stored back by every launch) ----
  L.xyz = take(3);
  L.vel = take(3);
  L.rpy = L.omega = L.quat = L.omega_world = -1;
  if (physics == PDX_PHYSICS_SIMPLE) {
    L.rpy = take(3);
    L.omega = take(3);
  } else {
    L.quat = take(4);
    L.omega_world = take(3);
  }
  L.motor_b = L.motor_k = L.motor_x = L.ring = L.ring_idx = -1;
  if (physics == PDX_PHYSICS_BULLET) {
    L.motor_x = take(4);
    L.ring = take(8);
    L.ring_idx = take(1);
  }
  L.ou = take(4);
  L.last_action = take(4);
  L.pid = pid ? take(12) : -1;
  L.ep_return = take(1);
  L.ep_length = take(1);
  L.ep_index = take(1);
  L.gyro_bias = L.gyro_lpf = -1;
  if (noise) {
    L.gyro_bias = take(3);
    L.gyro_lpf = take(3);
  }
  L.n_dyn_words = w;
  L.n_store_quads = (w + 3) / 4;
  // ---- per-episode constants (domain randomisation, circle offset): written by reset only.
  // They start in the padding of the last dynamic quad; quads holding only constants are
  // not stored by a step that does not reset.
  L.dt = take(1);
  L.mass = take(1);
  L.inertia = take(3);
  L.ftf1 = take(1);
  L.ref_offset = task == PDX_TASK_CIRCLE ? take(1) : -1;
  if (physics == PDX_PHYSICS_BULLET) {
    L.motor_b = take(4);
    L.motor_k = take(4);
  }
  L.n_words = w;
  L.n_quads = (w + 3) / 4;
  L.core_dim = core_dim_of(task, noise);
  L.hist_quads = (L.core_dim + 4 + 3) / 4;
  L.pack_quads = L.n_quads + (2 * L.core_dim + 3) / 4;
  return L;
}

// Image of pdx_policy_pack: the actor's net, then the critic's, each W1t[D][H], b1[H], W2t[H][H], b2[H], W3t[H][4],
// b3[4] with the hidden width zero padded to H.  k_policy stages the whole image, k_evaluate the actor's net.
// Words of one net, in the type of D: k_policy computes its shared-memory offsets in int, the ABI in int64_t.
template <class I>
constexpr I policy_net_words(I D, int H) { return D * H + H + H * H + H + H * 4 + 4; }
// H of the actor's net (the critic's is 64)
constexpr int policy_actor_pad(int h1, int h2) { return (h1 <= 52 && h2 <= 52) ? 52 : 64; }

// Tape slot counts (reference draw order; SURVEY 3.3 / A.5).
struct TapeSlots {
  int init, reset, step;
  int reset_task;      // draws of task_specific_reset
  int reset_dr;        // draws of apply_domain_randomization
  int obs_full;        // 33 when noise is on, else 0
  int obs_gyro;        // 9 / 0
};

inline TapeSlots tape_slots_of(const PdxConfig& c) {
  TapeSlots s{};
  const bool noise = c.observation_noise != 0;
  s.obs_full = noise ? 33 : 0;
  s.obs_gyro = noise ? 9 : 0;
  s.init = s.obs_full;
  const int ring_words = 4 * c.buf_size;
  if (c.task == PDX_TASK_TAKEOFF) s.reset_task = c.reset_distribution ? 3 : 0;
  else s.reset_task = c.reset_distribution ? 14 + 4 + ring_words : 0;
  s.reset_dr = c.domain_randomization > 0 ? (c.use_motor_dynamics ? 15 : 7) : 0;
  s.reset = s.reset_task + s.reset_dr + 2 * s.obs_full;
  int st = 0;
  for (int k = 0; k < c.agg; ++k) st += 4 + ((k % c.obs_rate) == 0 ? s.obs_full : s.obs_gyro);
  s.step = st + s.obs_full;
  return s;
}

}  // namespace pdx
