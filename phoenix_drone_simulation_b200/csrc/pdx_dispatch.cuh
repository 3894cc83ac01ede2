// Host-side dispatch: PdxConfig -> DevCfg<T> and the (task, physics, noise, rng) template
// switch.  Included by one translation unit per arithmetic type / physics so that the
// float64 parity kernels can be compiled with -fmad=false and the build parallelised.
#pragma once
#include <cmath>
#include <cstdlib>
#include "pdx_host.h"
#include "pdx_kernels.cuh"

namespace pdx {

enum Kind { KIND_INIT = 0, KIND_RESET = 1, KIND_STEP = 2 };

struct LaunchArgs {
  const PdxConfig* cfg;
  const PdxBuffers* buf;
  const float* actions;
  const uint8_t* mask;
  uint64_t seed, counter;
  double* dump_step;
  double* dump_reset;
  double* dump_init;
  int n_steps;
  cudaStream_t stream;
};

template <class T>
static void fill_devcfg(const PdxConfig& p, DevCfg<T>& d) {
  const TapeSlots ts = tape_slots_of(p);
  d.history = p.history; d.agg = p.agg; d.obs_rate = p.obs_rate; d.use_latency = p.use_latency;
  d.buf_size = p.buf_size; d.use_motor_dynamics = p.use_motor_dynamics;
  d.reset_distribution = p.reset_distribution; d.ground_effect = p.ground_effect;
  d.max_episode_steps = p.max_episode_steps; d.core_dim = p.core_dim; d.obs_dim = p.obs_dim;
  d.control_mode = p.control_mode;
  d.dr_on = p.domain_randomization > 0 ? 1 : 0; d.reset_on_nonfinite = p.reset_on_nonfinite; d.auto_reset = p.auto_reset;
  d.slots_obs_full = ts.obs_full; d.slots_obs_gyro = ts.obs_gyro;
  d.slots_reset_task = ts.reset_task; d.slots_reset_dr = ts.reset_dr;
  d.slots_step = ts.step; d.slots_reset = ts.reset;
  d.dr = (T)p.domain_randomization; d.time_step = (T)p.time_step; d.mass = (T)p.mass;
  for (int k = 0; k < 3; ++k) {
    d.inertia[k] = (T)p.inertia[k]; d.target[k] = (T)p.target_pos[k];
    d.init_xyz[k] = (T)p.init_xyz[k]; d.drag[k] = (T)p.drag_coeff[k];
  }
  d.arm = (T)p.arm;
  d.gravity = (T)p.gravity; d.thrust2weight = (T)p.thrust2weight; d.max_thrust = (T)p.max_thrust;
  d.k_mass_dr = (T)p.k_mass_dr; d.ftf1 = (T)p.ftf1; d.hover_x = (T)p.hover_x;
  d.hover_action = (T)p.hover_action; d.motor_tc = (T)p.motor_time_constant;
  d.ou_theta = (T)p.ou_theta; d.ou_sigma = (T)p.ou_sigma; d.lpf_ratio = (T)p.lpf_ratio;
  d.pos_std = (T)p.pos_norm_std; d.pos_unif = (T)p.pos_unif_range; d.vel_std = (T)p.vel_norm_std;
  d.quat_std = (T)p.quat_norm_std; d.quat_unif = (T)p.quat_unif_range;
  d.gyro_pi = (T)p.gyro_pi; d.gyro_sigma_b = (T)p.gyro_sigma_b; d.gyro_rw = (T)p.gyro_random_walk;
  d.gyro_to = (T)p.gyro_turn_on;
  d.gyro_white = (T)std::sqrt(p.gyro_random_walk * p.gyro_random_walk + p.gyro_turn_on * p.gyro_turn_on);
  d.pen_action = (T)p.penalty_action; d.pen_angle = (T)p.penalty_angle; d.pen_spin = (T)p.penalty_spin;
  d.pen_terminal = (T)p.penalty_terminal; d.pen_velocity = (T)p.penalty_velocity;
  d.arp = (T)p.action_rate_penalty;
  for (int k = 0; k < 4; ++k) { d.prop_xy[k][0] = (T)p.prop_xy[k][0]; d.prop_xy[k][1] = (T)p.prop_xy[k][1]; }
  d.prop_z = (T)p.prop_z; d.gec = (T)p.gnd_eff_coeff; d.prop_r = (T)p.prop_radius;
  d.ge_hclip = (T)p.gnd_eff_h_clip; d.lin_damp = (T)p.lin_damping; d.ang_damp = (T)p.ang_damping;
  d.ground_z = (T)p.ground_z;
}

// Launch shape of k_rollout for a shard of n environments on `sms` SMs: threads per block and one or two
// observation tiles.  The kernel runs at 128 registers, so an SM holds 16 warps whatever the block size.
//   * A shard that fits in one wave (every block resident at once; the block scheduler spreads them breadth
//     first): blocks of 128 to 512 threads, the shape with the fewest warps on the busiest SM.  A launch
//     lasts as long as its busiest SM, and the next launch waits for all of it.  65,536 environments in
//     128-thread blocks are 512 blocks on 148 SMs, 68 SMs with 16 warps and 80 with 12; in 448-thread blocks
//     they are one block of 14 warps per SM (measured on a B200: 393.6 -> 378.1 us per 64-step launch).
//   * A larger shard: blocks of 128, 64 or 32 threads, the most warps resident per SM under the
//     shared-memory plan.
// Ties go to the larger block, then to double buffering.  A one-wave shard never takes blocks of fewer than 128
// threads: their warps vote on package regeneration in groups of one to three and drift apart (measured at
// 65,536 environments, where they balance as well as 448 threads: 64 threads 538 us, 32 threads 963 us per launch).
struct LaunchShape { int block, tiles; size_t smem; };
template <class T>
static LaunchShape pick_shape(int D, int E, int wmode, int64_t n, int sms) {
  LaunchShape best{0, 0, 0}, best_wave{0, 0, 0};
  int best_warps = -1;
  int64_t best_busiest = -1;
  for (int block = 512; block >= 32; block -= 32) {
    const bool classic = block == 128 || block == 64 || block == 32;
    for (int tiles = 2; tiles >= 1; --tiles) {
      const size_t smem = rollout_smem_bytes<T>(block, D, tiles, E, wmode);
      if (smem > kMaxSmemBytes) continue;
      const int by_smem = (int)(((size_t)228 * 1024) / (smem + 1024));
      const int by_regs = 65536 / (128 * block);
      const int per_sm = by_smem < by_regs ? by_smem : by_regs;
      if (per_sm == 0) continue;
      const int warps = per_sm * (block / 32);
      if (classic && warps > best_warps) { best_warps = warps; best = LaunchShape{block, tiles, smem}; }
      const int64_t grid = (n + block - 1) / block;
      if (block < 128 || grid > (int64_t)per_sm * sms) continue;
      const int64_t busiest = (grid + sms - 1) / sms * (block / 32);
      if (best_busiest < 0 || busiest < best_busiest) { best_busiest = busiest; best_wave = LaunchShape{block, tiles, smem}; }
    }
  }
  return best_busiest >= 0 ? best_wave : best;
}

template <class T, int TASK, int PHYS, bool NOISE, int RNG, bool PID>
static cudaError_t launch_kind(int kind, const KArgs<T>& ka, cudaStream_t st) {
  const int64_t n = ka.b.n_envs;
  if (kind != KIND_STEP) {
    const int block = 128;
    const unsigned grid = (unsigned)((n + block - 1) / block);
    if (kind == KIND_INIT) k_init<T, TASK, PHYS, NOISE, RNG, PID><<<grid, block, 0, st>>>(ka);
    else k_reset<T, TASK, PHYS, NOISE, RNG, PID><<<grid, block, 0, st>>>(ka);
    return cudaGetLastError();
  }
  // row mode of the observation tiles (rollout_smem_bytes): 2 = padded rows, 128-bit history shift -- float32 rows of
  // whole 16-byte entries (Circle / TakeOff; measured: TakeOff H = 2 12.1 -> 14.4 G, Circle H = 8 2.75 -> 5.68 G
  // env-steps/s); 1 = rotated walk for the other D % 16 == 0
  typedef Model<T, TASK, PHYS, NOISE, RNG, PID> Mo;
  constexpr bool quad_ok = sizeof(T) == 4 && Mo::E % 4 == 0 && Mo::C % 4 == 0;
  int wmode = (ka.c.obs_dim & 15) == 0 ? (quad_ok ? 2 : 1) : 0;
  // PDX_WMODE forces mode 1 or 2 where legal: the tests run mode 1 as the reference of mode 2, switching the
  // variable between two environments of one process (so it is read per launch)
  if (const char* e = getenv("PDX_WMODE")) {
    const int wv = atoi(e);
    if (wmode && (wv == 1 || (wv == 2 && quad_ok))) wmode = wv;
  }
  int sms = 0;
  const cudaError_t es = sm_count(ka.b.device, &sms);
  if (es != cudaSuccess) return es;
  const LaunchShape shape = pick_shape<T>(ka.c.obs_dim, ka.c.core_dim + 4, wmode, n, sms);
  if (shape.block == 0) return cudaErrorInvalidConfiguration;
  KArgs<T> kb = ka;
  kb.n_tiles = shape.tiles;
  auto kern = wmode == 1 ? k_rollout<T, TASK, PHYS, NOISE, RNG, PID, 1> : k_rollout<T, TASK, PHYS, NOISE, RNG, PID, 0>;
  if constexpr (quad_ok) { if (wmode == 2) kern = k_rollout<T, TASK, PHYS, NOISE, RNG, PID, 2>; }
  const cudaError_t e = opt_in_smem(kern, ka.b.device, shape.smem);
  if (e != cudaSuccess) return e;
  const unsigned grid = (unsigned)((n + shape.block - 1) / shape.block);
  // early launch only on request (PDX_BUF_STATE_STABLE): measured, early launch of this kernel AND of a one-CTA-per-SM
  // tensor-core policy kernel around it collapses throughput (profiles/r1_summary.md), so the caller decides
  return launch_early(kern, grid, shape.block, shape.smem, st, (ka.b.flags & PDX_BUF_STATE_STABLE) != 0, kb);
}

template <class T, int TASK, int PHYS, bool PID>
static cudaError_t launch_nr(int kind, bool noise, int rng, const KArgs<T>& ka, cudaStream_t st) {
  if (noise) {
    if (rng == PDX_RNG_PHILOX) return launch_kind<T, TASK, PHYS, true, PDX_RNG_PHILOX, PID>(kind, ka, st);
    return launch_kind<T, TASK, PHYS, true, PDX_RNG_TAPE, PID>(kind, ka, st);
  }
  if (rng == PDX_RNG_PHILOX) return launch_kind<T, TASK, PHYS, false, PDX_RNG_PHILOX, PID>(kind, ka, st);
  return launch_kind<T, TASK, PHYS, false, PDX_RNG_TAPE, PID>(kind, ka, st);
}

// Kernel arguments of a finalised config and its buffers, with no actions, mask or dump tapes and one observation tile.
template <class T>
static KArgs<T> make_kargs(const PdxConfig& cfg, const PdxBuffers& buf, uint64_t seed, uint64_t counter, int n_steps) {
  KArgs<T> ka;
  fill_devcfg<T>(cfg, ka.c);
  ka.b = buf;
  ka.actions = nullptr; ka.mask = nullptr; ka.seed = seed; ka.counter = counter;
  ka.dump_step = ka.dump_reset = ka.dump_init = nullptr;
  ka.n_steps = n_steps; ka.n_tiles = 1;
  return ka;
}

// One arithmetic type, physics flavour and control family per translation unit.
template <class T, int PHYS, bool PID>
static cudaError_t launch_tu(int kind, const LaunchArgs& la) {
  KArgs<T> ka = make_kargs<T>(*la.cfg, *la.buf, la.seed, la.counter, la.n_steps);
  ka.actions = la.actions; ka.mask = la.mask;
  ka.dump_step = la.dump_step; ka.dump_reset = la.dump_reset; ka.dump_init = la.dump_init;
  ka.n_tiles = 2;
  const bool noise = la.cfg->observation_noise != 0;
  // pdx_dump_draws runs the TAPE-mode kernels with dump pointers set.
  const int rng = (la.dump_step || la.dump_reset || la.dump_init) ? PDX_RNG_TAPE : la.cfg->rng_mode;
  switch (la.cfg->task) {
    case PDX_TASK_HOVER: return launch_nr<T, PDX_TASK_HOVER, PHYS, PID>(kind, noise, rng, ka, la.stream);
    case PDX_TASK_CIRCLE: return launch_nr<T, PDX_TASK_CIRCLE, PHYS, PID>(kind, noise, rng, ka, la.stream);
    default: return launch_nr<T, PDX_TASK_TAKEOFF, PHYS, PID>(kind, noise, rng, ka, la.stream);
  }
}

// Implemented in pdx_tu_*.cu
cudaError_t launch_f32_simple(int kind, const LaunchArgs& la);
cudaError_t launch_f32_bullet(int kind, const LaunchArgs& la);
cudaError_t launch_f64_simple(int kind, const LaunchArgs& la);
cudaError_t launch_f64_bullet(int kind, const LaunchArgs& la);
cudaError_t launch_f32_simple_pid(int kind, const LaunchArgs& la);
cudaError_t launch_f32_bullet_pid(int kind, const LaunchArgs& la);
cudaError_t launch_f64_simple_pid(int kind, const LaunchArgs& la);
cudaError_t launch_f64_bullet_pid(int kind, const LaunchArgs& la);

}  // namespace pdx
