// pdx_evaluate: deterministic evaluation of P policies on E shared episodes in ONE launch
// (EnvironmentEvaluator.eval, utils/evaluation.py:52-107, for many policies at once).
//
//   for t in 0..max_episode_steps-1:   a = mu(standardise(obs))              (core.py:282-289, actor mean)
//                                      obs, r, terminated, truncated = env.step(a)   (no auto-reset)
//                                      while alive: ret += r, cost += c, len += 1
//
// Design
//   * one thread per (policy, episode); a block serves episodes of one policy only, the grid runs over
//     (policy, episode chunk).  The environment state stays in registers for the whole episode and steps
//     through rollout_step (pdx_kernels.cuh), the step body of k_rollout and k_collect, compiled with its
//     per-step global stores off: the step hands reward, cost and flags back through StepCtx.
//   * shared episodes: policy p's copy of the state is the block's StepCtx state with n = E, i = e, so the
//     environment draws are keyed by env_offset + e for every policy (common random numbers).
//   * the block stages its policy's actor image (the actor part of pdx_policy_pack) once.  The actor is
//     k_policy's arithmetic (pdx_rollout.cu: run_net / dense) operation for operation: each output starts from
//     its bias and takes one fma per input in input order, then relu.  This unit is built with -use_fast_math
//     (FTZ, approximate division) and pdx_rollout.cu is not, so the actor is written with explicit
//     round-to-nearest PTX without .ftz: its result does not depend on the unit's flags.
//   * the block stops as soon as every one of its episodes is over (block vote per step).
//
// Global traffic: the actor image and normaliser once per block, the initial state and observation once per
// episode, 20 bytes of results per episode (plus the optional validation records).
#include "pdx_dispatch.cuh"

namespace pdx {

constexpr int kEvChunk = 16;                  // actor outputs accumulated at a time (registers)

struct EvalArgs {
  int32_t P, E, D, h1, h2, HP, n_steps, blocks_per_policy;
  int64_t stride;                             // floats between two policies' images in `packed`
  int64_t quads;                              // state planes of one policy's copy
  const float* packed;                        // [P][stride]
  const float* mean; const float* std;        // [P][D] or NULL
  float eps;
  const float* obs0;                          // [E][D]
  float* state;                               // [P][quads][E][4]
  double* ret; double* cost; int32_t* len;    // [P][E]
  float* rec_obs; float* rec_act; float* rec_rew; float* rec_cost;   // optional [T][P][E](x D, x 4)
  uint8_t* rec_term; uint8_t* rec_trunc;
};

__device__ __forceinline__ float ev_fma(float a, float b, float c) {
  float d;
  asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float ev_sub(float a, float b) {
  float d;
  asm("sub.rn.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ float ev_mul(float a, float b) {
  float d;
  asm("mul.rn.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ float ev_relu(float a) {          // fmaxf(a, 0) without flushing subnormals
  float d;
  asm("max.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(0.0f));
  return d;
}

// shared-memory plan (bytes): norm float2 [D], actor image [policy_net_words], rows [B][D], hidden columns [HP][B]
__host__ __device__ inline size_t eval_smem_bytes(int B, int D, int HP) {
  const size_t norm = ((size_t)D * 8 + 15) & ~(size_t)15;
  return norm + (size_t)policy_net_words((int64_t)D, HP) * 4 + (size_t)B * D * 4 + (size_t)HP * B * 4;
}

// out[j] = b[j] + sum_i w[i][j] x_i for the kEvChunk outputs starting at w / b (row stride HP), in input order
template <class F>
__device__ __forceinline__ void ev_dense(const float* __restrict__ w, const float* __restrict__ b, int HP, int n_in, F in,
                                         float (&acc)[kEvChunk]) {
#pragma unroll
  for (int j = 0; j < kEvChunk; ++j) acc[j] = b[j];
  for (int i = 0; i < n_in; ++i) {
    const float x = in(i);
    const float4* row = reinterpret_cast<const float4*>(w + i * HP);
#pragma unroll
    for (int j4 = 0; j4 < kEvChunk / 4; ++j4) {
      const float4 wv = row[j4];
      acc[4 * j4 + 0] = ev_fma(wv.x, x, acc[4 * j4 + 0]);
      acc[4 * j4 + 1] = ev_fma(wv.y, x, acc[4 * j4 + 1]);
      acc[4 * j4 + 2] = ev_fma(wv.z, x, acc[4 * j4 + 2]);
      acc[4 * j4 + 3] = ev_fma(wv.w, x, acc[4 * j4 + 3]);
    }
  }
}

// actor mean of this thread's row (image layout of k_pack_policy: W1t[D][HP], b1, W2t[HP][HP], b2, W3t[HP][4], b3[4]).
// Chunks past h1 / h2 are skipped: their outputs are padding that the next layer never reads.
__device__ __forceinline__ float4 ev_actor(const float* __restrict__ img, const float2* __restrict__ norm, bool stdz,
                                           const float* __restrict__ row, float* __restrict__ hid, int D, int HP, int h1,
                                           int h2, int B, int tid) {
  const float* w1 = img;
  const float* b1 = w1 + D * HP;
  const float* w2 = b1 + HP;
  const float* b2 = w2 + HP * HP;
  const float* w3 = b2 + HP;
  const float* b3 = w3 + HP * 4;
  float acc[kEvChunk];
  for (int c0 = 0; c0 < h1; c0 += kEvChunk) {
    ev_dense(w1 + c0, b1 + c0, HP, D, [&](int i) {
      const float o = row[i];
      if (!stdz) return o;
      const float2 nm = norm[i];
      return ev_mul(ev_sub(o, nm.x), nm.y);
    }, acc);
#pragma unroll
    for (int j = 0; j < kEvChunk; ++j)
      if (c0 + j < h1) hid[(c0 + j) * B + tid] = ev_relu(acc[j]);
  }
  float mu[4] = {b3[0], b3[1], b3[2], b3[3]};
  for (int c0 = 0; c0 < h2; c0 += kEvChunk) {
    ev_dense(w2 + c0, b2 + c0, HP, h1, [&](int i) { return hid[i * B + tid]; }, acc);
#pragma unroll
    for (int j = 0; j < kEvChunk; ++j) {
      if (c0 + j < h2) {                      // layer 3 takes its inputs in order as they come out of layer 2
        const float y = ev_relu(acc[j]);
        const float4 wv = reinterpret_cast<const float4*>(w3)[c0 + j];
        mu[0] = ev_fma(wv.x, y, mu[0]); mu[1] = ev_fma(wv.y, y, mu[1]);
        mu[2] = ev_fma(wv.z, y, mu[2]); mu[3] = ev_fma(wv.w, y, mu[3]);
      }
    }
  }
  return make_float4(mu[0], mu[1], mu[2], mu[3]);
}

template <int TASK, int PHYS, bool NOISE, bool PID>
__global__ void __maxnreg__(168) k_evaluate(const __grid_constant__ KArgs<float> a, const __grid_constant__ EvalArgs p) {
  typedef float T;
  typedef Model<T, TASK, PHYS, NOISE, PDX_RNG_PHILOX, PID> Mo;
  const DevCfg<T>& c = a.c;
  const int B = blockDim.x, tid = threadIdx.x;
  const int D = p.D, HP = p.HP, E = p.E;
  const int pol = blockIdx.x / p.blocks_per_policy;
  const int e = (blockIdx.x % p.blocks_per_policy) * B + tid;
  const bool valid = e < E;
  const bool stdz = p.std != nullptr;

  extern __shared__ __align__(16) unsigned char smem[];
  float2* norm = reinterpret_cast<float2*>(smem);
  float* img = reinterpret_cast<float*>(smem + (((size_t)D * 8 + 15) & ~(size_t)15));
  const int64_t piw = policy_net_words((int64_t)D, HP);
  float* tile = img + piw;
  float* hid = tile + (size_t)B * D;
  // normaliser as k_policy stages it: (mean, 1 / (std + eps)), correctly rounded
  if (stdz) {
    for (int k = tid; k < D; k += B) {
      float s, inv;
      asm("add.rn.f32 %0, %1, %2;" : "=f"(s) : "f"(p.std[(int64_t)pol * D + k]), "f"(p.eps));
      asm("div.rn.f32 %0, %1, %2;" : "=f"(inv) : "f"(1.0f), "f"(s));
      norm[k] = make_float2(p.mean[(int64_t)pol * D + k], inv);
    }
  }
  {
    const float4* src = reinterpret_cast<const float4*>(p.packed + (int64_t)pol * p.stride);
    float4* dst = reinterpret_cast<float4*>(img);
    for (int64_t k = tid; k < piw / 4; k += B) dst[k] = src[k];
  }
  float* my_row = tile + (size_t)tid * D;
  T* state = p.state + (int64_t)pol * p.quads * E * 4;
  Mo m(c);
#pragma unroll
  for (int k = 0; k < Mo::NW; ++k) m.w[k] = T(0);
  if (valid) {
    m.load(state, E, e);
    for (int k = 0; k < D; ++k) my_row[k] = p.obs0[(int64_t)e * D + k];
  } else {
    for (int k = 0; k < D; ++k) my_row[k] = 0.0f;
  }
  __syncthreads();
  StepCtx<T> sc;
  sc.state = state; sc.n = E; sc.i = e; sc.valid = valid; sc.lane = tid & 31; sc.tid = tid; sc.B = B;
  sc.row0 = my_row; sc.row1 = my_row; sc.stg = nullptr; sc.RS = D; sc.acc_sum = nullptr; sc.acc_ext = nullptr; sc.NT = 1;
  sc.fast2 = false; sc.bulk = false; sc.latency = Mo::BULLET && c.use_latency; sc.any_fin = false;

  double ret = 0.0, cost = 0.0;
  int len = 0;
  bool alive = valid;
  for (int t = 0; t < p.n_steps; ++t) {
    const float4 mu = ev_actor(img, norm, stdz, my_row, hid, D, HP, p.h1, p.h2, B, tid);
    const int64_t r = ((int64_t)t * p.P + pol) * E + e;        // record index [t][pol][e]
    if (p.rec_obs && valid) {
      for (int k = 0; k < D; ++k) p.rec_obs[r * D + k] = my_row[k];
      reinterpret_cast<float4*>(p.rec_act)[r] = mu;
    }
    rollout_step<T, TASK, PHYS, NOISE, PDX_RNG_PHILOX, PID, 0, true>(a, m, sc, t, mu, [](bool) { return false; });
    if (alive) {
      ret += (double)sc.ev_reward;
      cost += (double)sc.ev_cost;
      len += 1;
      alive = !(sc.ev_terminated || sc.ev_truncated);
    }
    if (p.rec_obs && valid) {
      p.rec_rew[r] = sc.ev_reward; p.rec_cost[r] = sc.ev_cost;
      p.rec_term[r] = sc.ev_terminated ? 1 : 0; p.rec_trunc[r] = sc.ev_truncated ? 1 : 0;
    }
    // finished and padding threads keep stepping until the whole block is done
    if (!__syncthreads_or(alive)) break;
  }
  if (valid) {
    const int64_t o = (int64_t)pol * E + e;
    p.ret[o] = ret;
    p.cost[o] = cost;
    p.len[o] = len;
  }
}

// Threads per block: the candidate with the most resident warps for this grid (occupancy from the compiled
// kernel's registers and the shared-memory plan: wide rows shrink the block), ties to the smaller block (finer
// early exit, less tail).
template <int TASK, int PHYS, bool NOISE, bool PID>
static cudaError_t launch_evaluate(const KArgs<float>& ka, EvalArgs& p, int sms, cudaStream_t st) {
  auto kern = k_evaluate<TASK, PHYS, NOISE, PID>;
  int best_b = 0;
  int64_t best_warps = -1;
  for (int B = 32; B <= 256; B *= 2) {
    const size_t smem = eval_smem_bytes(B, p.D, p.HP);
    if (smem > kMaxSmemBytes) break;
    cudaError_t e = opt_in_smem(kern, ka.b.device, smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, B, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) break;
    const int64_t blocks = (int64_t)p.P * ((p.E + B - 1) / B);
    const int64_t resident = (blocks < (int64_t)per_sm * sms ? blocks : (int64_t)per_sm * sms) * (B / 32);
    if (resident > best_warps) { best_warps = resident; best_b = B; }
  }
  if (best_b == 0) return cudaErrorInvalidConfiguration;
  const size_t smem = eval_smem_bytes(best_b, p.D, p.HP);
  p.blocks_per_policy = (p.E + best_b - 1) / best_b;
  kern<<<(unsigned)((int64_t)p.P * p.blocks_per_policy), best_b, smem, st>>>(ka, p);
  return cudaGetLastError();
}

template <int TASK, int PHYS, bool PID>
static cudaError_t launch_evaluate_noise(bool noise, const KArgs<float>& ka, EvalArgs& p, int sms, cudaStream_t st) {
  return noise ? launch_evaluate<TASK, PHYS, true, PID>(ka, p, sms, st) : launch_evaluate<TASK, PHYS, false, PID>(ka, p, sms, st);
}

template <int TASK>
static cudaError_t launch_evaluate_task(const PdxConfig& c, const KArgs<float>& ka, EvalArgs& p, int sms, cudaStream_t st) {
  const bool noise = c.observation_noise != 0, pid = c.control_mode != PDX_CTRL_PWM;
  if (c.physics == PDX_PHYSICS_BULLET)
    return pid ? launch_evaluate_noise<TASK, PDX_PHYSICS_BULLET, true>(noise, ka, p, sms, st)
               : launch_evaluate_noise<TASK, PDX_PHYSICS_BULLET, false>(noise, ka, p, sms, st);
  return pid ? launch_evaluate_noise<TASK, PDX_PHYSICS_SIMPLE, true>(noise, ka, p, sms, st)
             : launch_evaluate_noise<TASK, PDX_PHYSICS_SIMPLE, false>(noise, ka, p, sms, st);
}

}  // namespace pdx

extern "C" int pdx_evaluate(const PdxConfig* cfg, const PdxBuffers* buf, const PdxPolicySet* set, const PdxEvaluation* out,
                            uint64_t seed, uint64_t counter, void* stream) {
  using namespace pdx;
  if (!cfg || !buf || !set || !out) return set_error(PDX_ERR_INVALID, "pdx_evaluate: null argument");
  PdxConfig c = *cfg;
  if (pdx_config_finalize(&c)) return PDX_ERR_INVALID;
  if (c.dtype != PDX_DTYPE_F32 || c.rng_mode != PDX_RNG_PHILOX)
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: supports float32 environments with Philox draws");
  const int64_t P = set->n_policies, E = set->episodes;
  if (P < 1 || E < 1 || P * E >= ((int64_t)1 << 31))
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: n_policies and episodes must be >= 1 with n_policies * episodes < 2^31");
  if (buf->n_envs != E || !buf->state || !buf->obs)
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: buf needs n_envs == episodes, state [P][quads][E][4] and obs [E][obs_dim]");
  if (set->obs_dim != c.obs_dim || set->hidden[0] < 1 || set->hidden[0] > 64 || set->hidden[1] < 1 || set->hidden[1] > 64 ||
      set->n_out < 1 || set->n_out > 4)
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: actor must match obs_dim, with two hidden layers of <= 64 units and <= 4 outputs");
  const int HP = policy_actor_pad(set->hidden[0], set->hidden[1]);
  if (!set->packed || set->stride < policy_net_words((int64_t)c.obs_dim, HP) || (set->stride & 3) || (!set->mean) != (!set->std))
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: packed images of pdx_policy_pack (stride >= the actor's words, a multiple of 4) "
                                      "and mean / std both given or both NULL are required");
  const bool rec = out->rec_obs || out->rec_act || out->rec_reward || out->rec_cost || out->rec_terminated || out->rec_truncated;
  if (!out->ret || !out->cost || !out->length ||
      (rec && !(out->rec_obs && out->rec_act && out->rec_reward && out->rec_cost && out->rec_terminated && out->rec_truncated)))
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: ret / cost / length are required, the record buffers all or none");
  if (eval_smem_bytes(32, c.obs_dim, HP) > kMaxSmemBytes)
    return set_error(PDX_ERR_INVALID, "pdx_evaluate: obs_dim too wide for the shared-memory plan");
  const int rc = select_device(buf->device);
  if (rc) return rc;
  c.auto_reset = 0;                                           // an evaluation episode is not reset
  KArgs<float> ka = make_kargs<float>(c, *buf, seed, counter, c.max_episode_steps);
  ka.b.obs = ka.b.reward = ka.b.cost = ka.b.final_obs = ka.b.episode_return = nullptr;
  ka.b.terminated = ka.b.truncated = nullptr; ka.b.episode_length = nullptr; ka.b.episode_stats = nullptr;
  ka.b.tape_step = ka.b.tape_reset = ka.b.tape_init = nullptr;
  EvalArgs p;
  p.P = (int32_t)P; p.E = (int32_t)E; p.D = c.obs_dim; p.h1 = set->hidden[0]; p.h2 = set->hidden[1]; p.HP = HP;
  p.n_steps = c.max_episode_steps; p.blocks_per_policy = 1;
  p.stride = set->stride; p.quads = pdx_state_quads(&c);
  p.packed = set->packed; p.mean = set->mean; p.std = set->std; p.eps = set->eps;
  p.obs0 = reinterpret_cast<const float*>(buf->obs); p.state = reinterpret_cast<float*>(buf->state);
  p.ret = out->ret; p.cost = out->cost; p.len = out->length;
  p.rec_obs = out->rec_obs; p.rec_act = out->rec_act; p.rec_rew = out->rec_reward; p.rec_cost = out->rec_cost;
  p.rec_term = out->rec_terminated; p.rec_trunc = out->rec_truncated;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, buf->device);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  if (c.task == PDX_TASK_HOVER) e = launch_evaluate_task<PDX_TASK_HOVER>(c, ka, p, sms, st);
  else if (c.task == PDX_TASK_CIRCLE) e = launch_evaluate_task<PDX_TASK_CIRCLE>(c, ka, p, sms, st);
  else e = launch_evaluate_task<PDX_TASK_TAKEOFF>(c, ka, p, sms, st);
  return cuda_error("pdx_evaluate", e);
}
