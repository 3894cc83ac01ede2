/*
 * phoenix_b200.h -- C ABI of the B200-native batched Crazyflie stepping engine.
 *
 * Drop-in boundary for the env-step hot path of SvenGronauer/phoenix-drone-simulation
 * (paths below are relative to the reference's phoenix_drone_simulation/ package).
 * The reference has no FFI of its own for this path (it is pure Python calling the
 * PyBullet C extension); the entry points below are what a `ctypes` binding inside the
 * reference's `DroneBaseEnv` would bind to replace
 *     envs/base.py:382-431   DroneBaseEnv.reset
 *     envs/base.py:433-475   DroneBaseEnv.step            (+ everything it calls:
 *         envs/physics.py:91-200, envs/agents.py:259-298, envs/control.py:94-100,
 *         envs/sensors.py:75-134, envs/utils.py:32-108, envs/{hover,circle,takeoff}.py)
 *     algs/core.py:458-534   Buffer.finish_path / discount_cumsum (GAE)
 *     utils/online_mean_std.py:50-95 and utils/mpi_tools.py:217-240 (the moment sums
 *         that feed the cross-rank all-reduce)
 * INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *  - Every buffer is caller-allocated DEVICE memory (PyTorch tensors in practice) passed
 *    as raw pointers + sizes.  The library allocates nothing persistent and keeps no
 *    pointers between calls; all constants travel in PdxConfig (kernel parameter space).
 *  - All launches go to the caller-supplied stream and never synchronise.
 *  - Return value: 0 on success, negative PdxStatus otherwise; pdx_last_error() returns a
 *    thread-local message.  Nothing throws across the ABI.
 *  - There is NO CPU fallback: without a CUDA device every compute entry point fails.
 *  - Random numbers are counter based (Philox4x32-10 keyed by `seed`, indexed by the
 *    GLOBAL env index, the caller's `counter` and a per-draw-site id), so results do not
 *    depend on how environments are sharded over GPUs and there is no library-side
 *    mutable state.
 */
#ifndef PHOENIX_B200_H_
#define PHOENIX_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDX_ABI_VERSION 7

typedef enum PdxStatus {
  PDX_OK = 0,
  PDX_ERR_INVALID = -1,       /* bad argument / unsupported configuration */
  PDX_ERR_CUDA = -2,          /* CUDA runtime error (message in pdx_last_error) */
  PDX_ERR_NO_DEVICE = -3      /* no CUDA device: there is no CPU path */
} PdxStatus;

enum { PDX_TASK_HOVER = 0, PDX_TASK_CIRCLE = 1, PDX_TASK_TAKEOFF = 2 };   /* envs/{hover,circle,takeoff}.py */
enum { PDX_PHYSICS_SIMPLE = 0, PDX_PHYSICS_BULLET = 1 };                  /* envs/physics.py:127 / :79 */
enum { PDX_DTYPE_F32 = 0, PDX_DTYPE_F64 = 1 };
enum { PDX_RNG_PHILOX = 0, PDX_RNG_TAPE = 1 };
enum { PDX_CTRL_PWM = 0, PDX_CTRL_ATTITUDE_RATE = 1, PDX_CTRL_ATTITUDE = 2 };         /* envs/control.py:91,120,194 */
enum { PDX_MAX_HISTORY = 16 };

/* Persistent per-environment state lives in `state` as 16-byte "quads" (4 x real), one
 * plane per quad: quad q of env i is at  state + (q * n_envs + i) * 4 * sizeof(real),
 * so a warp's access to one quad is one contiguous 512-byte (f32) segment (128-bit
 * per-thread accesses).  Quad/lane assignment: pdx_state_field(). */

typedef struct PdxConfig {
  /* ---- structure ------------------------------------------------------------------ */
  int32_t task;                 /* PDX_TASK_*                                             */
  int32_t physics;              /* PDX_PHYSICS_*   (physics string, base.py:222-230)      */
  int32_t dtype;                /* PDX_DTYPE_*: arithmetic + state/obs/reward storage type */
  int32_t rng_mode;             /* PDX_RNG_*                                              */
  int32_t observation_noise;    /* 1 if observation_noise > 0          (base.py:130)      */
  int32_t history;              /* observation_history_size H >= 1     (base.py:44)       */
  int32_t agg;                  /* aggregate_phy_steps                 (base.py:35,457)   */
  int32_t obs_rate;             /* sim_freq // observation_frequency   (base.py:108)      */
  int32_t use_latency;          /* agents.py:165                                          */
  int32_t buf_size;             /* latency ring length, agents.py:180  (1 or 2 supported) */
  int32_t use_motor_dynamics;   /* agents.py:196                                          */
  int32_t reset_distribution;   /* enable_reset_distribution           (base.py:38)       */
  int32_t ground_effect;        /* physics.py:18 (never enabled by the reference)         */
  int32_t max_episode_steps;    /* TimeLimit, __init__.py:11 (500)                        */
  int32_t core_dim;             /* C: width of one compute_observation()                  */
  int32_t obs_dim;              /* D = H * (C + 4)                     (base.py:143)      */
  int32_t reset_on_nonfinite;   /* extension: treat a non-finite state as truncation      */
  int32_t auto_reset;           /* 1: an env whose episode ends is reset inside pdx_step  */
  int32_t control_mode;         /* PDX_CTRL_*  (control_mode string, agents.py:71-78)       */
  int32_t reserved_i[1];
  /* ---- scalars (all double; converted once per launch) --------------------------- */
  double domain_randomization;  /* p of U(v(1-p), v(1+p)); <= 0 disables (base.py:259)    */
  double time_step;             /* TIME_STEP = 1/sim_freq              (base.py:98)       */
  double sensor_dt;             /* 1/SIM_FREQ handed to SensorNoise    (hover.py:144)     */
  double mass;                  /* M, urdf                                                */
  double inertia[3];            /* IXX, IYY, IZZ, urdf                                    */
  double arm;                   /* L: torque arm, (x*L)/sqrt(2)        (physics.py:167)   */
  double gravity;               /* 9.81 (agents.py:145, physics.py:16)                    */
  double thrust2weight;         /* urdf                                                   */
  double max_thrust;            /* K without DR: G*M*T2W/4             (agents.py:149,200)*/
  double k_mass_dr;             /* 0.028: hard-coded mass of K under DR (agents.py:224)   */
  double ftf0, ftf1;            /* force-torque factors                (agents.py:142-143)*/
  double hover_x, hover_action; /* agents.py:152-153                                      */
  double motor_time_constant;   /* base.py:41                                             */
  double ou_theta, ou_sigma;    /* envs/utils.py:88, agents.py:206                        */
  double lpf_ratio;             /* gyro LPF Ts/T = 0.5                 (base.py:109-110)  */
  double pos_norm_std, pos_unif_range, vel_norm_std;            /* sensors.py:20-23       */
  double quat_norm_std, quat_unif_range;                        /* sensors.py:24-25       */
  double gyro_pi, gyro_sigma_b, gyro_random_walk, gyro_turn_on; /* sensors.py:121-134     */
  double penalty_action, penalty_angle, penalty_spin, penalty_terminal, penalty_velocity;
  double action_rate_penalty;   /* ARP (hover.py:28, circle.py:28)                        */
  double target_pos[3];         /* hover.py:14                                            */
  double init_xyz[3];           /* hover.py:44, takeoff.py:51 (float32-quantised values)  */
  double drag_coeff[3];         /* urdf drag_coeff_xy/_z               (agents.py:252-254)*/
  double prop_xy[4][2];         /* propeller joint origins, cf21x_bullet.urdf:59-136      */
  double prop_z;                /* 0.0108 (bullet) / 0 (sys_eq)                           */
  double gnd_eff_coeff, prop_radius, gnd_eff_h_clip;            /* agents.py:156,250-251  */
  double lin_damping, ang_damping;  /* btMultiBody defaults 0.04 (third-party, unpinned)  */
  double ground_z;              /* half height of the collision cylinder (Bullet ids)     */
  double reserved_d[8];
} PdxConfig;

/* PdxBuffers.flags.  The step kernels are launched with programmatic stream serialisation (sm_90+):
 * a launch may start while the kernel before it on the stream drains, and waits (griddepcontrol.wait)
 * before it touches anything that kernel could have written.  PDX_BUF_STATE_STABLE is the caller's
 * promise that the kernel launched immediately before this one on the stream does NOT write `state`
 * (the collector: the policy kernel sits between two env.step launches) -- the per-env state is then
 * loaded before the wait, under the predecessor's tail. */
#define PDX_BUF_STATE_STABLE 1

typedef struct PdxBuffers {
  int64_t n_envs;               /* environments in this shard, 1 .. 2^31 - 1              */
  int64_t env_offset;           /* global index of local env 0 (RNG subsequence)          */
  int32_t device;               /* CUDA device ordinal the buffers live on                */
  int32_t flags;                /* PDX_BUF_* bits, 0 = none                               */
  void*   state;                /* [pdx_state_quads][n_envs][4] real                      */
  void*   obs;                  /* out  [n_envs][obs_dim] real, row-major                 */
  void*   reward;               /* out  [n_envs] real                (step only)          */
  void*   cost;                 /* out  [n_envs] real                (step only)          */
  uint8_t* terminated;          /* out  [n_envs]                     (step only)          */
  uint8_t* truncated;           /* out  [n_envs]                     (step only)          */
  void*   final_obs;            /* out, optional: obs of the step that ended an episode   */
  void*   episode_return;       /* out, optional [n_envs] real: return of a finished ep.  */
  int32_t* episode_length;      /* out, optional [n_envs]                                 */
  double* episode_stats;        /* in/out, optional [8]: n, sum ret, sum ret^2, sum len,  */
                                /*   min ret, max ret, min len, max len (block-reduced)   */
  const double* tape_step;      /* PDX_RNG_TAPE: [step_slots][n_envs] standardised draws  */
  const double* tape_reset;     /* PDX_RNG_TAPE: [reset_slots][n_envs]                    */
  const double* tape_init;      /* PDX_RNG_TAPE: [33][n_envs] constructor observation     */
} PdxBuffers;

/* ---- queries (no device needed) ---------------------------------------------------- */
int         pdx_abi_version(void);
const char* pdx_last_error(void);
int         pdx_config_size(void);                       /* sizeof(PdxConfig)  */
int         pdx_buffers_size(void);                      /* sizeof(PdxBuffers) */
/* Validates a configuration; fills core_dim / obs_dim.  0 or PDX_ERR_INVALID. */
int         pdx_config_finalize(PdxConfig* cfg);
int         pdx_state_quads(const PdxConfig* cfg);       /* planes of 4 reals per env */
/* Location of a named state field ("xyz","vel","rpy","omega","quat","omega_world","dt",
 * "mass","inertia","ftf1","motor_a","motor_k","motor_x","ring","ring_idx","ou",
 * "gyro_bias","gyro_lpf","last_action","pid","ep_return","ep_length","ref_offset","hist").  Writes the first word index (quad*4+lane) and the
 * length in words; returns 0, or PDX_ERR_INVALID if the field does not exist. */
int         pdx_state_field(const PdxConfig* cfg, const char* name, int* first_word, int* n_words);
int         pdx_tape_slots(const PdxConfig* cfg, int* reset_slots, int* step_slots, int* init_slots);
/* Algorithmic HBM bytes per environment of one launch that advances n_steps env.steps: state and
 * history read once and written once, plus per step the action in and the observation row,
 * reward, cost and flags out.  pdx_step_bytes(cfg) == pdx_rollout_bytes(cfg, 1). */
int64_t     pdx_step_bytes(const PdxConfig* cfg);
int64_t     pdx_rollout_bytes(const PdxConfig* cfg, int32_t n_steps);

/* ---- compute (CUDA; fail with PDX_ERR_NO_DEVICE / PDX_ERR_CUDA otherwise) ------------- */
int pdx_device_count(void);
/* Constructor semantics (base.py:26-153): zero state, nominal parameters and the one
 * compute_observation() call of base.py:143 (seeds the gyro bias when noise is on). */
int pdx_init(const PdxConfig* cfg, const PdxBuffers* buf, uint64_t seed, uint64_t counter,
             void* stream);
/* DroneBaseEnv.reset for every env whose mask byte is non-zero (all if mask == NULL);
 * writes the first observation of the new episode to buf->obs. */
int pdx_reset(const PdxConfig* cfg, const PdxBuffers* buf, const uint8_t* mask,
              uint64_t seed, uint64_t counter, void* stream);
/* DroneBaseEnv.step for all envs in lock-step with in-kernel auto-reset: an env whose
 * episode ends (terminated, or max_episode_steps reached) is reset in the same launch and
 * buf->obs receives the first observation of its next episode.  `actions`: [n_envs][4]
 * float32 (the policy's dtype; the PWM stage quirk of control.py:98-99 depends on it). */
int pdx_step(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions,
             uint64_t seed, uint64_t counter, void* stream);
/* n_steps env.steps of every environment in ONE launch (the rollout-collector form of
 * roll_out's inner loop, algs/iwpg/iwpg.py:355-385, for open-loop action sequences): the state
 * stays in registers between steps.  `actions` is [n_steps][n_envs][4]; every per-step output of
 * PdxBuffers is time-major with n_steps leading: obs [n_steps][n_envs][obs_dim], reward / cost /
 * terminated / truncated / episode_return / episode_length [n_steps][n_envs], final_obs
 * [n_steps][n_envs][obs_dim]; tapes [n_steps][slots][n_envs].  Step t draws its random numbers
 * at `counter + t`, so the caller advances its counter by n_steps.  pdx_step == n_steps 1. */
int pdx_step_many(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions, int32_t n_steps,
                  uint64_t seed, uint64_t counter, void* stream);
/* Debug/validation: runs pdx_init (init_tape != NULL), pdx_reset of all envs (actions ==
 * NULL, reset_tape != NULL) or pdx_step (actions != NULL; needs step_tape and reset_tape) with
 * the production Philox draws and additionally writes every draw consumed into tape layout
 * ([slots][n_envs] doubles), so that the CPU oracle can replay exactly what the kernel used. */
int pdx_dump_draws(const PdxConfig* cfg, const PdxBuffers* buf, const float* actions,
                   uint64_t seed, uint64_t counter,
                   double* step_tape, double* reset_tape, double* init_tape, void* stream);

/* ---- rollout collector pieces (algs/core.py, utils/online_mean_std.py) ----------------- */
/* GAE over a [T][n] rollout laid out time-major, one thread per env column, reverse scan
 * with episode boundaries (Buffer.finish_path, core.py:497-534, incl. the reward-scaling
 * quirk that also scales the appended bootstrap value).  All float32.
 *   rew,val,done(uint8: 1 = terminated, 2 = truncated/cut -> bootstrap with boot_val)
 *   boot_val [T][n]: V(next obs) where done==2 (ignored elsewhere); last_val [n]: V after T
 *   outputs adv, target_v, disc_ret: [T][n].
 *   Reward scaling (use_reward_scaling != 0) divides by `ret_scale`, or by *ret_std_dev + ret_scale when
 *   ret_std_dev (DEVICE pointer to the running std of the returns, online_mean_std.py:42-48) is not
 *   NULL -- ret_scale then carries the epsilon; the collector never reads the std back to the host. */
int pdx_gae(int64_t T, int64_t n, const float* rew, const float* val, const uint8_t* done,
            const float* boot_val, const float* last_val, float gamma, float lam,
            float ret_scale, int use_reward_scaling, const float* ret_std_dev,
            float* adv, float* target_v, float* disc_ret, void* stream);
/* Column moments of x [rows][dim] (float32, row-major): out[0..dim) += sum x,
 * out[dim..2dim) += sum (x-shift)^2 with shift[dim] (NULL = 0); doubles.  Feeds the
 * OnlineMeanStd all-reduce. */
int pdx_moments(int64_t rows, int32_t dim, const float* x, const double* shift,
                double* out, void* stream);

/* OnlineMeanStd.update (utils/online_mean_std.py:70-95) from the column sums of pdx_moments / pdx_collect, in place on
 * the device: s1[dim] = sum (x - shift), s2[dim] = sum (x - shift)^2 over `rows` local rows (shift NULL = 0); `world`
 * ranks with equal batch sizes.  Single rank: phase 3.  Several ranks (the reference averages the batch mean and the
 * batch second moment over the ranks, mpi_tools.py:199-214): phase 0 writes batch_mean[dim] -> caller all-reduces it
 * to the rank average -> phase 1 writes batch_var[dim] -> caller averages it -> phase 2 updates mean / std / count. */
int pdx_oms_update(int32_t dim, const double* s1, const double* s2, double rows, int32_t world, const float* shift,
                   float* batch_mean, float* batch_var, float* mean, float* std, float* count, int32_t phase,
                   void* stream);

/* ActorCritic.step (algs/core.py:370-393) fused into one launch: standardise the observation
 * ((o - mean) / (std + eps), utils/online_mean_std.py:42-48; std == NULL skips it), Gaussian actor
 * MLP (two hidden layers, relu), critic MLP (two hidden layers, tanh), a = mu + exp(log_std) * N(0,1)
 * drawn with Philox keyed by (seed, env index, counter), log-probability.  Weights are torch
 * nn.Linear tensors ([out][in] row-major float32) on the device; hidden sizes <= 64, n_out <= 4.
 * obs [n][obs_dim] float32; actions [n][4], values [n], logp [n], mu_out [n][4] (optional). */
typedef struct PdxMlp {
  int32_t hidden[2];
  int32_t n_out;
  int32_t reserved;
  const float* weight[3];
  const float* bias[3];
} PdxMlp;
/* `packed`: device buffer of pdx_policy_pack_words() floats holding the weights transposed and zero
 * padded as the kernel stages them; refresh it with pdx_policy_pack after every weight update. */
int64_t pdx_policy_pack_words(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v);
int pdx_policy_pack(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, float* packed, void* stream);
/* `env_offset`: global index of row 0 -- the action noise is keyed by the GLOBAL environment index, like the
 * environment's own draws, so a rollout does not depend on how the environments are sharded over GPUs. */
int pdx_policy_step(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                    const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, uint64_t seed,
                    uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp, float* mu_out,
                    void* stream);

/* The same ActorCritic.step (algs/core.py:370-393; MLPGaussianActor core.py:227-289, MLPCritic core.py:297-310,
 * standardisation utils/online_mean_std.py:42-48) on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators
 * and hidden activations in tensor memory; csrc/pdx_policy_tc.cu).  128 environments per tile, one
 * persistent CTA per SM (two for precision 1).  `precision`: 1 = operands rounded to TF32 once
 * (~1e-3 relative error on mu / value), 3 = split-TF32 (hi + lo operands, three products per term):
 * float32-level results.  Same Philox draws as pdx_policy_step for the same (seed, counter, env).
 * Needs its own packed image (pdx_policy_tc_pack_words / pdx_policy_tc_pack; refresh after every
 * weight update).  PDX_ERR_INVALID if the shapes do not fit (hidden > 64, n_out > 4, obs_dim too
 * wide for the shared-memory plan): callers then use pdx_policy_step.
 * `precision | PDX_POLICY_TC_OVERLAP`: the caller promises that the kernel launched immediately before on
 * the stream writes none of the weight image / normaliser / log_std (the collector: an env.step launch),
 * so the kernel stages them while that kernel drains (programmatic dependent launch). */
#define PDX_POLICY_TC_OVERLAP 0x100
int64_t pdx_policy_tc_pack_words(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, int32_t precision);
int pdx_policy_tc_pack(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, int32_t precision, float* packed, void* stream);
int pdx_policy_step_tc(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                       const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, int32_t precision,
                       uint64_t seed, uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp,
                       float* mu_out, void* stream);

/* ---- the fused collector step: IWPGAlgorithm.roll_out's loop (algs/iwpg/iwpg.py:350-385) in ONE launch ----
 * For T = rollout->n_steps steps and every environment of the shard:
 *     a, v, logp = ActorCritic.step(obs)            (algs/core.py:370-393, the networks of `policy`)
 *     obs, r, terminated, truncated = env.step(a)   (envs/base.py:433-475, in-kernel auto-reset)
 * followed by last_val = V(obs) (the value that bootstraps the cut at the end of the rollout, iwpg.py:376-378).
 * The environment state stays in registers for the whole rollout and the policy networks run on the tensor
 * cores (tcgen05, accumulators and hidden activations in tensor memory) between two env.steps of the same
 * thread; csrc/pdx_collect.cu.  Outputs are time-major: buf->obs [T][n][obs_dim] receives the observation
 * AFTER step t (row t + 1 of a [T+1][n][obs_dim] rollout tensor whose row 0 is rollout->obs0), buf->reward /
 * cost / terminated / truncated [T][n], buf->final_obs (optional) [T][n][obs_dim], buf->episode_stats.
 * Step t draws the environment noise at `counter + t` (as pdx_step_many) and the action noise at
 * policy->counter + t with the Philox stream of pdx_policy_step_tc keyed by the GLOBAL environment index.
 * Supported: float32, Philox, observation noise on, PWM control, the Hover and Circle ids (obs_dim <= 64 and not a
 * multiple of 16), auto_reset, two hidden layers of <= 64 units with the actor's first layer <= 63 (the kernel
 * appends a constant-1 unit that carries the layer-2 biases through the MMAs); PDX_ERR_INVALID otherwise (callers
 * then alternate pdx_policy_step_tc and pdx_step). */
typedef struct PdxPolicy {
  int32_t obs_dim;
  int32_t precision;            /* 1 = single-TF32 operands (float32 data, low 13 mantissa bits dropped by the tensor core), */
                                /* 3 = split TF32 (float32-level results)                                                    */
  const float* mean;            /* observation normaliser (utils/online_mean_std.py:42-48); std == NULL skips it */
  const float* std;
  float eps;
  int32_t reserved;
  const PdxMlp* pi;             /* Gaussian actor, two hidden layers (relu), <= 4 outputs */
  const PdxMlp* v;              /* critic, two hidden layers (tanh), 1 output */
  const float* log_std;         /* [n_out] */
  const float* packed;          /* weight image of pdx_policy_tc_pack for this precision */
  uint64_t seed, counter;       /* Philox key / position of the action noise */
} PdxPolicy;
typedef struct PdxRollout {
  int32_t n_steps;              /* T */
  int32_t reserved;
  const float* obs0;            /* [n][obs_dim] observation the rollout starts from */
  float* act;                   /* out [T][n][4] */
  float* val;                   /* out [T][n]    */
  float* logp;                  /* out [T][n]    */
  float* last_val;              /* out [n]: V(observation after the last step) */
  void*  scratch;               /* device scratch of at least pdx_collect_scratch_bytes(device) bytes */
  int64_t scratch_bytes;
  double* obs_moments;          /* in/out, optional [2][obs_dim]: += sum (o - mean), += sum (o - mean)^2 over the T x n  */
                                /* observations the policy saw (mean = policy->mean, 0 without normaliser): what         */
                                /* OnlineMeanStd.update needs (utils/online_mean_std.py:70-84), without a pass over obs  */
} PdxRollout;
int64_t pdx_collect_scratch_bytes(int32_t device);
int pdx_collect(const PdxConfig* cfg, const PdxBuffers* buf, const PdxPolicy* policy, const PdxRollout* rollout,
                uint64_t seed, uint64_t counter, void* stream);

/* ---- deterministic evaluation of many policies on shared episodes (utils/evaluation.py:52-107) ----
 * EnvironmentEvaluator.eval for P policies x E episodes in ONE launch (csrc/pdx_evaluate.cu): every policy acts
 * with its actor mean on the standardised observation (core.py:282-289) for at most max_episode_steps steps, without
 * auto-reset; an episode accumulates reward, cost and length up to and including the step that reports terminated
 * or truncated.  Episode e of every policy starts from the same state and sees the same draws (keyed by
 * buf->env_offset + e, step t at `counter + t` as pdx_step_many): the results of a policy do not depend on the
 * other policies of the call.  The actor arithmetic is pdx_policy_step's, bit for bit.
 *   buf: n_envs == episodes; state [P][pdx_state_quads][E][4], P copies of the state after pdx_init + pdx_reset of
 *        E environments; obs [E][obs_dim], the observation that pdx_reset returned.  The state is read, not written.
 * Supported: float32 with Philox draws, every task / physics / control mode, obs_dim up to the shared-memory plan
 * (history 16 included); PDX_ERR_INVALID otherwise, and for bad arguments before any device call. */
typedef struct PdxPolicySet {
  int32_t n_policies;           /* P >= 1 */
  int32_t episodes;             /* E >= 1, P * E < 2^31 */
  int32_t obs_dim;
  int32_t hidden[2];            /* actor hidden sizes (<= 64), the same for every policy */
  int32_t n_out;                /* actor outputs (<= 4); actions past n_out are 0 */
  int64_t stride;               /* floats between two images in `packed` (>= the actor part, a multiple of 4) */
  const float* packed;          /* [P][stride]: pdx_policy_pack images; only the actor part is read */
  const float* mean;            /* [P][obs_dim] observation normaliser, or NULL (with std) for none */
  const float* std;             /* [P][obs_dim] */
  float eps;                    /* (o - mean) / (std + eps) */
  int32_t reserved;
} PdxPolicySet;
typedef struct PdxEvaluation {
  double* ret;                  /* out [P][E] episode return  */
  double* cost;                 /* out [P][E] episode cost    */
  int32_t* length;              /* out [P][E] episode length  */
  /* optional validation records, all or none, [T][P][E] with T = max_episode_steps; steps after every episode of
   * a block ended are not written */
  float* rec_obs;               /* [T][P][E][obs_dim] observation the actor saw */
  float* rec_act;               /* [T][P][E][4] action */
  float* rec_reward;            /* [T][P][E] */
  float* rec_cost;              /* [T][P][E] */
  uint8_t* rec_terminated;      /* [T][P][E] */
  uint8_t* rec_truncated;       /* [T][P][E] */
} PdxEvaluation;
int pdx_evaluate(const PdxConfig* cfg, const PdxBuffers* buf, const PdxPolicySet* set, const PdxEvaluation* out,
                 uint64_t seed, uint64_t counter, void* stream);

/* ---- PPO update: losses and exact gradients of one network (algs/ppo/ppo.py:22-40, algs/iwpg/iwpg.py:398-485) ----
 * csrc/pdx_ppo.cu, CUDA cores, float32 with float64 cross-CTA sums.  Weights come straight from the torch nn.Linear
 * tensors through PdxMlp; gradients are written into caller tensors of the same shapes (p.grad), the loss as a float32
 * device scalar.  Networks: two hidden layers of <= 64 units; obs_dim 1 .. 384.
 *   pdx_ppo_pi_grad, actor (relu, 4 outputs, log_std fixed: it gets no gradient), per sample i of the batch:
 *     mu = pi(obs), logp = sum_j (-((a - mu) / std)^2 / 2 - log_std - log(2 pi) / 2), r = exp(logp - logp_old),
 *     loss = -mean(min(r A, clip(r, 1 - clip_ratio, 1 + clip_ratio) A)); d loss / d logp = -r A / n where
 *     r A <= clip(r) A and 0 elsewhere (torch's minimum / clamp backward).  grad == NULL: forward only.  Optional
 *     mu [n][4] receives pi(obs); with mu_ref [n][4] (and kl) kl = mean_i sum_j (mu_ref - mu)^2 / (2 std^2), the
 *     Gaussian KL at equal std.
 *     clip_ratio = +INFINITY: no clip, loss = -mean(r A) (IWPG / NPG / TRPO's surrogate), d loss / d logp = -r A / n
 *     everywhere; a non-finite ratio makes the loss non-finite, as in torch.
 *   pdx_ppo_v_grad, critic (tanh, 1 output): loss = mean((v(obs) - target_v)^2).
 * Row i of the batch is index[i] (index NULL: i) of obs / act / adv / logp_old / target_v; mu / mu_ref are indexed
 * by i.  Indices must lie inside the caller's tensors (not checked).  scratch: device memory of
 * pdx_ppo_scratch_bytes(device, obs_dim, net) bytes (net->n_out 4 = actor, 1 = critic); a smaller one, down to one
 * CTA's partial sums, runs fewer CTAs.  Results are bit-identical from run to run for the same device, inputs and
 * scratch size (fixed assignment of samples to CTAs, fixed summation order).  PDX_ERR_INVALID for unsupported shapes
 * and bad arguments, before any device call. */
typedef struct PdxMlpGrad {
  float* weight[3];             /* [out][in], like PdxMlp.weight */
  float* bias[3];
} PdxMlpGrad;
typedef struct PdxPpoBatch {
  int64_t n;                    /* samples, >= 1 */
  int32_t obs_dim;
  int32_t reserved;
  const float* obs;             /* [rows][obs_dim] standardised observations */
  const int64_t* index;         /* optional [n]; NULL = rows 0 .. n-1 */
  const float* act;             /* [rows][4]  actor  */
  const float* adv;             /* [rows]     actor  */
  const float* logp_old;        /* [rows]     actor  */
  const float* target_v;        /* [rows]     critic */
} PdxPpoBatch;
int64_t pdx_ppo_scratch_bytes(int32_t device, int32_t obs_dim, const PdxMlp* net);
int pdx_ppo_pi_grad(const PdxPpoBatch* batch, const PdxMlp* pi, const float* log_std, float clip_ratio,
                    const PdxMlpGrad* grad, float* loss, float* mu, const float* mu_ref, float* kl,
                    void* scratch, int64_t scratch_bytes, void* stream);
int pdx_ppo_v_grad(const PdxPpoBatch* batch, const PdxMlp* v, const PdxMlpGrad* grad, float* loss,
                   void* scratch, int64_t scratch_bytes, void* stream);
/* Fisher-vector product of the actor (algs/npg/npg.py Fvp) for conjugate-gradient policy updates:
 *     out = scale * (1/n) sum_i J_i^T diag(std^-2) J_i dir + damping * dir,   J_i = d pi(obs_i) / d theta  [4 x params]
 * = scale x the Hessian of pdx_ppo_pi_grad's kl (mean over samples, sum over the 4 action dimensions) at the current
 * weights applied to dir, plus damping.  theta = the six nn.Linear tensors of `pi` (log_std is frozen and has no
 * entry); `dir` and `out` are shaped like them ([out][in] weights and biases, dir->hidden == pi->hidden, n_out 4), and
 * `out` must not overlap `dir`.  The batch uses n, obs_dim, obs and index only (every 4th row: pass an index).
 * scratch: pdx_ppo_scratch_bytes(device, obs_dim, pi) bytes.  Float32 per sample, float64 sums rounded once;
 * bit-identical from run to run like the gradients.  PDX_ERR_INVALID before any device call for the shapes
 * pdx_ppo_pi_grad rejects, a dir of another shape, missing pointers, non-finite scale, negative or non-finite damping
 * and a scratch smaller than one CTA's partials. */
int pdx_ppo_pi_fvp(const PdxPpoBatch* batch, const PdxMlp* pi, const float* log_std, const PdxMlp* dir,
                   float scale, float damping, const PdxMlpGrad* out, void* scratch, int64_t scratch_bytes,
                   void* stream);

/* Cross-rank combination of the 8-word episode statistics (utils/mpi_tools.py:217-240 does four
 * MPI all-reduces per key): the caller all-gathers the per-rank vectors into gathered[world][8]
 * (one NCCL call) and this writes out[0..4) = sums, out[4], out[6] = minima, out[5], out[7] = maxima. */
int pdx_stats_combine(int32_t world, const double* gathered, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* PHOENIX_B200_H_ */
