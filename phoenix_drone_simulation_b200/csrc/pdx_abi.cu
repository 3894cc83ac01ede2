// extern "C" entry points of libphoenix_b200.so (declared in include/phoenix_b200.h).
#include <cstdio>
#include <cstring>
#include <cmath>
#include "pdx_dispatch.cuh"

namespace {

thread_local char g_err[512] = "";
}  // namespace

int pdx::set_error(int code, const char* msg) {
  std::snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

namespace {

int fail(int code, const char* fmt, const char* detail = "") {
  std::snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}

pdx::Layout layout_of(const PdxConfig* c) {
  return pdx::make_layout(c->task, c->physics, c->observation_noise != 0, c->control_mode != PDX_CTRL_PWM);
}

int validate(const PdxConfig* c) {
  if (!c) return fail(PDX_ERR_INVALID, "null config");
  if (c->task < 0 || c->task > 2) return fail(PDX_ERR_INVALID, "bad task");
  if (c->physics < 0 || c->physics > 1) return fail(PDX_ERR_INVALID, "bad physics");
  if (c->dtype < 0 || c->dtype > 1) return fail(PDX_ERR_INVALID, "bad dtype");
  if (c->rng_mode < 0 || c->rng_mode > 1) return fail(PDX_ERR_INVALID, "bad rng_mode");
  if (c->control_mode < 0 || c->control_mode > 2) return fail(PDX_ERR_INVALID, "bad control_mode");
  if (c->history < 1 || c->history > PDX_MAX_HISTORY) return fail(PDX_ERR_INVALID, "observation_history_size must be in [1,16]");
  if (c->agg < 1 || c->agg > 8) return fail(PDX_ERR_INVALID, "aggregate_phy_steps must be in [1,8]");
  if (c->obs_rate < 1 || c->agg % c->obs_rate != 0)
    return fail(PDX_ERR_INVALID, "aggregate_phy_steps must be a multiple of sim_freq//observation_frequency");
  if (c->buf_size < 1 || c->buf_size > 2) return fail(PDX_ERR_INVALID, "latency ring length must be 1 or 2 sub-steps");
  if (c->use_latency && c->agg < c->buf_size)
    return fail(PDX_ERR_INVALID, "aggregate_phy_steps must be >= latency ring length");
  if (c->physics == PDX_PHYSICS_SIMPLE && (c->use_latency || c->use_motor_dynamics))
    return fail(PDX_ERR_INVALID, "latency / motor dynamics belong to the Bullet agent");
  if (c->max_episode_steps < 1) return fail(PDX_ERR_INVALID, "max_episode_steps must be >= 1");
  return PDX_OK;
}

int check_buffers(const PdxConfig* c, const PdxBuffers* b, bool step) {
  if (!b) return fail(PDX_ERR_INVALID, "null buffers");
  if (b->n_envs <= 0) return fail(PDX_ERR_INVALID, "n_envs must be positive");
  if (b->n_envs >= ((int64_t)1 << 31)) return fail(PDX_ERR_INVALID, "n_envs must be below 2^31 per shard");
  if (!b->state || !b->obs) return fail(PDX_ERR_INVALID, "state/obs buffers are required");
  if (step && (!b->reward || !b->cost || !b->terminated || !b->truncated))
    return fail(PDX_ERR_INVALID, "reward/cost/terminated/truncated buffers are required");
  return PDX_OK;
}

int launch(const char* what, int kind, const PdxConfig* cfg, const PdxBuffers* buf, const float* actions,
           const uint8_t* mask, uint64_t seed, uint64_t counter, double* ds, double* dr, double* di,
           void* stream, int n_steps = 1) {
  int rc = validate(cfg);
  if (rc) return rc;
  PdxConfig c = *cfg;
  pdx_config_finalize(&c);
  rc = check_buffers(&c, buf, kind == pdx::KIND_STEP);
  if (rc) return rc;
  const bool dumping = ds || dr || di;
  if (c.rng_mode == PDX_RNG_TAPE && !dumping) {
    const pdx::TapeSlots ts = pdx::tape_slots_of(c);
    if (kind == pdx::KIND_STEP && ((ts.step && !buf->tape_step) || (ts.reset && !buf->tape_reset)))
      return fail(PDX_ERR_INVALID, "tape mode needs tape_step and tape_reset");
    if (kind == pdx::KIND_RESET && ts.reset && !buf->tape_reset) return fail(PDX_ERR_INVALID, "tape mode needs tape_reset");
    if (kind == pdx::KIND_INIT && ts.init && !buf->tape_init) return fail(PDX_ERR_INVALID, "tape mode needs tape_init");
  }
  if (kind == pdx::KIND_STEP && !actions) return fail(PDX_ERR_INVALID, "null actions");
  if (kind == pdx::KIND_STEP && (n_steps < 1 || n_steps > (1 << 20))) return fail(PDX_ERR_INVALID, "n_steps must be in [1, 2^20]");
  rc = pdx::select_device(buf->device);
  if (rc) return rc;
  cudaError_t e;
  pdx::LaunchArgs la{&c, buf, actions, mask, seed, counter, ds, dr, di, n_steps, (cudaStream_t)stream};
  const bool pid = c.control_mode != PDX_CTRL_PWM, simple = c.physics == PDX_PHYSICS_SIMPLE;
  if (c.dtype == PDX_DTYPE_F32)
    e = simple ? (pid ? pdx::launch_f32_simple_pid(kind, la) : pdx::launch_f32_simple(kind, la))
               : (pid ? pdx::launch_f32_bullet_pid(kind, la) : pdx::launch_f32_bullet(kind, la));
  else
    e = simple ? (pid ? pdx::launch_f64_simple_pid(kind, la) : pdx::launch_f64_simple(kind, la))
               : (pid ? pdx::launch_f64_bullet_pid(kind, la) : pdx::launch_f64_bullet(kind, la));
  return pdx::cuda_error(what, e);
}

}  // namespace

extern "C" {

int pdx_abi_version(void) { return PDX_ABI_VERSION; }
const char* pdx_last_error(void) { return g_err; }
int pdx_config_size(void) { return (int)sizeof(PdxConfig); }
int pdx_buffers_size(void) { return (int)sizeof(PdxBuffers); }

int pdx_config_finalize(PdxConfig* cfg) {
  const int rc = validate(cfg);
  if (rc) return rc;
  cfg->core_dim = pdx::core_dim_of(cfg->task, cfg->observation_noise != 0);
  cfg->obs_dim = cfg->history * (cfg->core_dim + 4);
  return PDX_OK;
}

int pdx_state_quads(const PdxConfig* cfg) {
  if (validate(cfg)) return PDX_ERR_INVALID;
  const pdx::Layout L = layout_of(cfg);
  return L.n_quads + (cfg->history - 1) * L.hist_quads + pdx::kPackSlots * L.pack_quads;
}

int pdx_state_field(const PdxConfig* cfg, const char* name, int* first_word, int* n_words) {
  if (validate(cfg) || !name || !first_word || !n_words) return fail(PDX_ERR_INVALID, "bad argument");
  const pdx::Layout L = layout_of(cfg);
  struct F { const char* n; int off; int len; };
  const F fields[] = {
      {"xyz", L.xyz, 3}, {"vel", L.vel, 3}, {"rpy", L.rpy, 3}, {"omega", L.omega, 3},
      {"quat", L.quat, 4}, {"omega_world", L.omega_world, 3}, {"dt", L.dt, 1}, {"mass", L.mass, 1},
      {"inertia", L.inertia, 3}, {"ftf1", L.ftf1, 1}, {"motor_b", L.motor_b, 4},
      {"motor_k", L.motor_k, 4}, {"motor_x", L.motor_x, 4}, {"ring", L.ring, 8},
      {"ring_idx", L.ring_idx, 1}, {"ou", L.ou, 4}, {"last_action", L.last_action, 4}, {"pid", L.pid, 12},
      {"ep_return", L.ep_return, 1}, {"ep_length", L.ep_length, 1}, {"ep_index", L.ep_index, 1},
      {"pool", (L.n_quads + (cfg->history - 1) * L.hist_quads) * 4, pdx::kPackSlots * L.pack_quads * 4},
      {"ref_offset", L.ref_offset, 1}, {"gyro_bias", L.gyro_bias, 3}, {"gyro_lpf", L.gyro_lpf, 3},
      {"hist", L.n_quads * 4, (cfg->history - 1) * L.hist_quads * 4},
  };
  for (const F& f : fields) {
    if (std::strcmp(f.n, name) == 0) {
      if (f.off < 0) return fail(PDX_ERR_INVALID, "field '%s' does not exist in this configuration", name);
      *first_word = f.off;
      *n_words = f.len;
      return PDX_OK;
    }
  }
  return fail(PDX_ERR_INVALID, "unknown state field '%s'", name);
}

int pdx_tape_slots(const PdxConfig* cfg, int* reset_slots, int* step_slots, int* init_slots) {
  if (validate(cfg)) return PDX_ERR_INVALID;
  const pdx::TapeSlots ts = pdx::tape_slots_of(*cfg);
  if (reset_slots) *reset_slots = ts.reset;
  if (step_slots) *step_slots = ts.step;
  if (init_slots) *init_slots = ts.init;
  return PDX_OK;
}

int64_t pdx_step_bytes(const PdxConfig* cfg) { return pdx_rollout_bytes(cfg, 1); }

int64_t pdx_rollout_bytes(const PdxConfig* cfg, int32_t n_steps) {
  if (validate(cfg) || n_steps < 1) return PDX_ERR_INVALID;
  const pdx::Layout L = layout_of(cfg);
  const int64_t sz = cfg->dtype == PDX_DTYPE_F32 ? 4 : 8;
  const int64_t E = L.core_dim + 4, H = cfg->history;
  // per launch: state + history read once and written once; per step: action in, observation
  // row, reward, cost and the two flag bytes out.  The bookkeeping word of the reset-package pool
  // (ep_index) and the pool itself are this implementation's, not the algorithm's: not counted.
  const int64_t words = L.n_words - 1;
  const int64_t once = (words + (H - 1) * E) * sz + (words + (H - 1) * E) * sz;
  const int64_t per_step = (H * E + 2) * sz + 16 + 2;
  return once + per_step * n_steps;
}

int pdx_device_count(void) {
  int n = 0;
  pdx::count_devices(&n);
  return n;
}

int pdx_init(const PdxConfig* cfg, const PdxBuffers* buf, uint64_t seed, uint64_t counter, void* stream) {
  return launch("pdx_init", pdx::KIND_INIT, cfg, buf, nullptr, nullptr, seed, counter, nullptr, nullptr, nullptr, stream);
}

int pdx_reset(const PdxConfig* cfg, const PdxBuffers* buf, const uint8_t* mask, uint64_t seed,
              uint64_t counter, void* stream) {
  return launch("pdx_reset", pdx::KIND_RESET, cfg, buf, nullptr, mask, seed, counter, nullptr, nullptr, nullptr, stream);
}

int pdx_step(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions, uint64_t seed,
             uint64_t counter, void* stream) {
  return launch("pdx_step", pdx::KIND_STEP, cfg, buf, actions, nullptr, seed, counter, nullptr, nullptr, nullptr, stream);
}

int pdx_step_many(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions, int32_t n_steps,
                  uint64_t seed, uint64_t counter, void* stream) {
  return launch("pdx_step_many", pdx::KIND_STEP, cfg, buf, actions, nullptr, seed, counter, nullptr, nullptr, nullptr, stream, n_steps);
}

}  // extern "C"

// pdx_dump_draws: run init / reset / step with the Philox draws copied out in tape layout.
extern "C" int pdx_dump_draws(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions,
                              uint64_t seed, uint64_t counter, double* step_tape, double* reset_tape,
                              double* init_tape, void* stream) {
  if (init_tape)
    return launch("pdx_dump_draws", pdx::KIND_INIT, cfg, buf, nullptr, nullptr, seed, counter, nullptr, nullptr, init_tape, stream);
  if (!actions && reset_tape)
    return launch("pdx_dump_draws", pdx::KIND_RESET, cfg, buf, nullptr, nullptr, seed, counter, nullptr, reset_tape, nullptr, stream);
  if (actions && step_tape && reset_tape)
    return launch("pdx_dump_draws", pdx::KIND_STEP, cfg, buf, actions, nullptr, seed, counter, step_tape, reset_tape, nullptr, stream);
  return fail(PDX_ERR_INVALID, "pdx_dump_draws: inconsistent tape pointers");
}
