// Rollout-collector kernels: GAE reverse scan and column moments.
//   pdx_gae     restates Buffer.finish_path / calculate_adv_and_value_targets /
//               discount_cumsum (algs/core.py:105-119, 458-479, 497-534) for a lock-step
//               [T][n] rollout: one thread per environment column walks time backwards and
//               restarts the recursions at episode boundaries.
//   pdx_moments restates the per-rank sums behind OnlineMeanStd.update
//               (utils/online_mean_std.py:70-84): sum x and sum (x - shift)^2 per column.
//   *_members   the same (and the fused policy step) for the P members of a population, blockIdx.y = member.
#include "pdx_host.h"
#include "pdx_layout.h"
#include "pdx_math.cuh"

namespace {

// column i of a [T][n] rollout
__device__ __forceinline__ void gae_column(int64_t i, int64_t T, int64_t n, const float* __restrict__ rew,
                                           const float* __restrict__ val, const uint8_t* __restrict__ done,
                                           const float* __restrict__ boot_val, const float* __restrict__ last_val,
                                           float gamma, float lam, float ret_scale, int use_scaling,
                                           float* __restrict__ adv, float* __restrict__ target_v,
                                           float* __restrict__ disc_ret) {
  float next_val = last_val[i];       // epoch cut: bootstrap with V(o_T)        (iwpg.py:376-378)
  float next_ret = next_val;          // rews = [..., last_val]                   (core.py:514)
  float next_adv = 0.0f;
  // The recurrence is serial in t but its loads are not: they are issued kChunk steps at a time (the scan is a
  // chain of L2 / HBM round trips otherwise: 57 us -> 22 us per 65,536 x 64 rollout)
  constexpr int kChunk = 8;
  for (int64_t t0 = T; t0 > 0; t0 -= kChunk) {
    uint8_t d[kChunk];
    float r[kChunk], v[kChunk];
#pragma unroll
    for (int u = 0; u < kChunk; ++u) {
      const int64_t t = t0 - 1 - u;
      if (t >= 0) { const int64_t k = t * n + i; d[u] = done[k]; r[u] = rew[k]; v[u] = val[k]; }
    }
#pragma unroll
    for (int u = 0; u < kChunk; ++u) {
      const int64_t t = t0 - 1 - u;
      if (t < 0) break;
      const int64_t k = t * n + i;
      if (d[u] == 1) { next_val = 0.0f; next_ret = 0.0f; next_adv = 0.0f; }          // terminated: v = 0
      else if (d[u] == 2) { next_val = boot_val[k]; next_ret = next_val; next_adv = 0.0f; }  // time limit
      const float ret = r[u] + gamma * next_ret;                                   // core.py:518
      float rs = r[u];
      if (use_scaling) rs = fminf(fmaxf(r[u] / ret_scale, -10.0f), 10.0f);         // core.py:527, oms clip
      const float delta = rs + gamma * next_val - v[u];                            // core.py:464
      const float a = delta + gamma * lam * next_adv;                              // core.py:465
      disc_ret[k] = ret;
      adv[k] = a;
      target_v[k] = a + v[u];                                                      // core.py:466
      next_val = v[u]; next_ret = ret; next_adv = a;
    }
  }
}

__global__ void __launch_bounds__(128) k_gae(int64_t T, int64_t n, const float* __restrict__ rew,
                                             const float* __restrict__ val, const uint8_t* __restrict__ done,
                                             const float* __restrict__ boot_val, const float* __restrict__ last_val,
                                             float gamma, float lam, float ret_scale, int use_scaling,
                                             const float* __restrict__ ret_std_dev,
                                             float* __restrict__ adv, float* __restrict__ target_v,
                                             float* __restrict__ disc_ret) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (ret_std_dev) ret_scale += ret_std_dev[0];     // running std of the returns, read on the device (no host sync)
  gae_column(i, T, n, rew, val, done, boot_val, last_val, gamma, lam, ret_scale, use_scaling, adv, target_v, disc_ret);
}

// k_gae over the [T][P * N] rollout of a population: column i belongs to member i / N and scales its rewards by that
// member's running return std ret_std_dev[i / N]
__global__ void __launch_bounds__(128) k_gae_members(int64_t T, int64_t n, int64_t N, const float* __restrict__ rew,
                                                     const float* __restrict__ val, const uint8_t* __restrict__ done,
                                                     const float* __restrict__ boot_val, const float* __restrict__ last_val,
                                                     float gamma, float lam, float ret_scale, int use_scaling,
                                                     const float* __restrict__ ret_std_dev,
                                                     float* __restrict__ adv, float* __restrict__ target_v,
                                                     float* __restrict__ disc_ret) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (ret_std_dev) ret_scale += ret_std_dev[i / N];
  gae_column(i, T, n, rew, val, done, boot_val, last_val, gamma, lam, ret_scale, use_scaling, adv, target_v, disc_ret);
}

// blockDim = (cols padded to 32, rows per block); each block strides over row tiles; row r is at x + row(r)
template <class Row>
__device__ __forceinline__ void moments_body(int64_t rows, int dim, Row row, const double* __restrict__ shift,
                                             double* __restrict__ out) {
  extern __shared__ double sm[];                     // [2][blockDim.y][blockDim.x]
  const int d = threadIdx.x;
  double s1 = 0.0, s2 = 0.0;
  if (d < dim) {
    const double sh = shift ? shift[d] : 0.0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.y + threadIdx.y; r < rows; r += (int64_t)gridDim.x * blockDim.y) {
      const double v = (double)row(r)[d];
      s1 += v;
      s2 += (v - sh) * (v - sh);
    }
  }
  const int idx = threadIdx.y * blockDim.x + d;
  sm[idx] = s1;
  sm[blockDim.x * blockDim.y + idx] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && d < dim) {
    for (int y = 1; y < blockDim.y; ++y) {
      s1 += sm[y * blockDim.x + d];
      s2 += sm[blockDim.x * blockDim.y + y * blockDim.x + d];
    }
    atomicAdd(&out[d], s1);
    atomicAdd(&out[dim + d], s2);
  }
}

__global__ void k_moments(int64_t rows, int dim, const float* __restrict__ x,
                          const double* __restrict__ shift, double* __restrict__ out) {
  moments_body(rows, dim, [=](int64_t r) { return x + r * dim; }, shift, out);
}

// member blockIdx.y of a [T][P * N][dim] population rollout: its T * N rows, shift [P][dim], out [P][2 dim]
__global__ void k_moments_members(int64_t T, int64_t N, int dim, const float* __restrict__ x,
                                  const double* __restrict__ shift, double* __restrict__ out) {
  const int64_t m = blockIdx.y, PN = (int64_t)gridDim.y * N;
  moments_body(T * N, dim, [=](int64_t r) { return x + ((r / N) * PN + m * N + r % N) * dim; },
               shift ? shift + m * dim : shift, out + 2 * m * dim);
}

// Combines the episode-statistics vectors of all ranks after one all-gather:
// out[0..4) = column sums, out[4], out[6] = column minima, out[5], out[7] = column maxima.
__global__ void k_stats_combine(int world, const double* __restrict__ gathered, double* __restrict__ out) {
  const int k = threadIdx.x;
  if (k >= 8) return;
  double v = gathered[k];
  for (int r = 1; r < world; ++r) {
    const double x = gathered[r * 8 + k];
    v = k < 4 ? v + x : ((k & 1) ? fmax(v, x) : fmin(v, x));
  }
  out[k] = v;
}

// OnlineMeanStd.update (utils/online_mean_std.py:70-95) from column sums, one thread per column.  The reference's
// algebra, including its rank averages: phase 0 writes the local batch mean (float32), phase 1 -- after the caller
// averaged it over the ranks -- the local batch second moment about the NEW mean, phase 2 -- after the second
// average -- updates mean / std / count in place; phase 3 = all three at once for a single rank.
__global__ void k_oms_update(int dim, const double* __restrict__ s1, const double* __restrict__ s2, double rows, double world,
                             const float* __restrict__ shift, float* __restrict__ bmean, float* __restrict__ bvar,
                             float* __restrict__ mean, float* __restrict__ std, float* __restrict__ count, int phase) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (phase == 4) {                 // the count is shared by all columns: bumped by a launch of its own, after the update
    if (d == 0) count[0] = count[0] + (float)(rows * world);
    return;
  }
  if (d < dim) {
    const double c = shift ? (double)shift[d] : 0.0;
    const double S1 = s1[d] + rows * c, S2 = s2[d] + 2.0 * c * s1[d] + rows * c * c;      // sums of x, x^2
    const float n_A = count[0], n_B = (float)(rows * world), n_AB = n_A + n_B;
    if (phase == 0 || phase == 3) bmean[d] = (float)(S1 / rows);
    if (phase == 0) return;
    const float delta = bmean[d] - mean[d];
    const float mean_new = mean[d] + delta * n_B / n_AB;
    if (phase == 1 || phase == 3) {
      const double mm = (double)mean_new;
      bvar[d] = (float)fmax((S2 - 2.0 * mm * S1 + rows * mm * mm) / rows, 0.0);
    }
    if (phase == 1) return;
    const float M2 = n_A * std[d] * std[d] + n_B * bvar[d] + delta * delta * (n_A * n_B / n_AB);
    mean[d] = mean_new;
    std[d] = sqrtf(M2 / n_AB);
  }
}

}  // namespace

extern "C" int pdx_gae(int64_t T, int64_t n, const float* rew, const float* val, const uint8_t* done,
                       const float* boot_val, const float* last_val, float gamma, float lam,
                       float ret_scale, int use_reward_scaling, const float* ret_std_dev, float* adv, float* target_v,
                       float* disc_ret, void* stream) {
  if (T <= 0 || n <= 0) return pdx::set_error(PDX_ERR_INVALID, "pdx_gae: T and n must be positive");
  if (!rew || !val || !done || !boot_val || !last_val || !adv || !target_v || !disc_ret)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_gae: null buffer");
  const int rc = pdx::select_device_of(rew);
  if (rc) return rc;
  const unsigned grid = (unsigned)((n + 127) / 128);
  k_gae<<<grid, 128, 0, (cudaStream_t)stream>>>(T, n, rew, val, done, boot_val, last_val, gamma, lam,
                                                ret_scale, use_reward_scaling, ret_std_dev, adv, target_v, disc_ret);
  return pdx::cuda_error("pdx_gae", cudaGetLastError());
}

extern "C" int pdx_moments(int64_t rows, int32_t dim, const float* x, const double* shift, double* out,
                           void* stream) {
  if (rows <= 0 || dim <= 0 || dim > 1024) return pdx::set_error(PDX_ERR_INVALID, "pdx_moments: rows must be positive and dim in [1, 1024]");
  if (!x || !out) return pdx::set_error(PDX_ERR_INVALID, "pdx_moments: null buffer");
  const int rc = pdx::select_device_of(x);
  if (rc) return rc;
  // blockDim = (dim, rows per block): thread (y, x) reads x[row * dim + x], so the linear thread id
  // walks the row-major matrix contiguously -- every lane of every warp is busy whatever dim is
  const int bx = dim;
  const int by = bx >= 256 ? 1 : 256 / bx;
  const dim3 block(bx, by);
  int64_t tiles = (rows + by - 1) / by;
  const unsigned grid = (unsigned)(tiles < 2368 ? tiles : 2368);      // 16 x 148 SMs
  const size_t smem = 2ull * bx * by * sizeof(double);
  k_moments<<<grid, block, smem, (cudaStream_t)stream>>>(rows, dim, x, shift, out);
  return pdx::cuda_error("pdx_moments", cudaGetLastError());
}

extern "C" int pdx_gae_members(int32_t members, int64_t T, int64_t n, const float* rew, const float* val,
                               const uint8_t* done, const float* boot_val, const float* last_val, float gamma, float lam,
                               float ret_scale, int use_reward_scaling, const float* ret_std_dev, float* adv,
                               float* target_v, float* disc_ret, void* stream) {
  if (members < 1 || T <= 0 || n <= 0 || n > INT64_MAX / members)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_gae_members: members, T and n must be positive");
  if (!rew || !val || !done || !boot_val || !last_val || !adv || !target_v || !disc_ret)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_gae_members: null buffer");
  const int rc = pdx::select_device_of(rew);
  if (rc) return rc;
  const int64_t cols = members * n;
  const unsigned grid = (unsigned)((cols + 127) / 128);
  k_gae_members<<<grid, 128, 0, (cudaStream_t)stream>>>(T, cols, n, rew, val, done, boot_val, last_val, gamma, lam,
                                                        ret_scale, use_reward_scaling, ret_std_dev, adv, target_v, disc_ret);
  return pdx::cuda_error("pdx_gae_members", cudaGetLastError());
}

extern "C" int pdx_moments_members(int32_t members, int64_t T, int64_t n, int32_t dim, const float* x,
                                   const double* shift, double* out, void* stream) {
  if (members < 1 || members > 65535 || T <= 0 || n <= 0 || dim <= 0 || dim > 1024)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_moments_members: members in [1, 65535], T and n positive, dim in [1, 1024]");
  if (!x || !out) return pdx::set_error(PDX_ERR_INVALID, "pdx_moments_members: null buffer");
  const int rc = pdx::select_device_of(x);
  if (rc) return rc;
  // pdx_moments' block shape; the row tiles of the whole launch stay within 16 x 148 SMs' worth of blocks
  const int bx = dim;
  const int by = bx >= 256 ? 1 : 256 / bx;
  const int64_t tiles = (T * n + by - 1) / by;
  const int64_t cap = (2368 + members - 1) / members;
  const dim3 grid((unsigned)(tiles < cap ? tiles : cap), (unsigned)members);
  const size_t smem = 2ull * bx * by * sizeof(double);
  k_moments_members<<<grid, dim3(bx, by), smem, (cudaStream_t)stream>>>(T, n, dim, x, shift, out);
  return pdx::cuda_error("pdx_moments_members", cudaGetLastError());
}

extern "C" int pdx_oms_update(int32_t dim, const double* s1, const double* s2, double rows, int32_t world, const float* shift,
                              float* batch_mean, float* batch_var, float* mean, float* std, float* count, int32_t phase,
                              void* stream) {
  if (dim <= 0 || !s1 || !s2 || rows <= 0 || world < 1 || !batch_mean || !batch_var || !mean || !std || !count || phase < 0 || phase > 3)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_oms_update: bad argument");
  const int rc = pdx::select_device_of(mean);
  if (rc) return rc;
  const unsigned grid = (unsigned)((dim + 127) / 128);
  k_oms_update<<<grid, 128, 0, (cudaStream_t)stream>>>(dim, s1, s2, rows, (double)world, shift, batch_mean, batch_var, mean, std, count, phase);
  if (phase >= 2)
    k_oms_update<<<1, 32, 0, (cudaStream_t)stream>>>(dim, s1, s2, rows, (double)world, shift, batch_mean, batch_var, mean, std, count, 4);
  return pdx::cuda_error("pdx_oms_update", cudaGetLastError());
}

extern "C" int pdx_stats_combine(int32_t world, const double* gathered, double* out, void* stream) {
  if (world <= 0 || !gathered || !out) return pdx::set_error(PDX_ERR_INVALID, "pdx_stats_combine: bad argument");
  const int rc = pdx::select_device_of(gathered);
  if (rc) return rc;
  k_stats_combine<<<1, 32, 0, (cudaStream_t)stream>>>(world, gathered, out);
  return pdx::cuda_error("pdx_stats_combine", cudaGetLastError());
}

// =============================================================================================
//  Fused policy step: ActorCritic.step (algs/core.py:370-393) for N environments in one launch:
//  observation standardisation (utils/online_mean_std.py:42-48), Gaussian actor MLP (two hidden
//  layers, relu; core.py:227-289), critic MLP (two hidden layers, tanh; core.py:297-310), action
//  sample a = mu + exp(log_std) * eps with on-device Philox draws, and log-probability.
//  One thread per environment.  Weights live in shared memory transposed to [in][out] so that a
//  warp reads them as 128-bit broadcasts; a layer streams its inputs one at a time (from global
//  memory for the first layer, from a per-thread shared column for the hidden ones) and keeps its
//  <= 64 output accumulators in registers.
// =============================================================================================
namespace {

constexpr int kPolBlock = 256;
constexpr int kHidMax = 64;

// tanh(x) = 1 - 2 / (exp(2x) + 1): two MUFU operations, ~1e-6 absolute error (tanhf costs ~30
// instructions and there are 128 activations per environment).
__device__ __forceinline__ float fast_tanh(float x) {
  const float e = __expf(2.0f * fminf(fmaxf(x, -15.0f), 15.0f));
  return 1.0f - __fdividef(2.0f, e + 1.0f);
}

// acc[j] += sum_i Wt[i][j] * x_i ; inputs x_i come from `in(i)`.
template <int OUT, class F>
__device__ __forceinline__ void dense(const float* __restrict__ wt, const float* __restrict__ bias, int n_in, F in,
                                      float (&acc)[OUT]) {
#pragma unroll
  for (int j = 0; j < OUT; ++j) acc[j] = bias[j];
  for (int i = 0; i < n_in; ++i) {
    const float x = in(i);
    const float4* row = reinterpret_cast<const float4*>(wt + i * OUT);
#pragma unroll
    for (int j4 = 0; j4 < OUT / 4; ++j4) {
      const float4 wv = row[j4];
      acc[4 * j4 + 0] = fmaf(wv.x, x, acc[4 * j4 + 0]);
      acc[4 * j4 + 1] = fmaf(wv.y, x, acc[4 * j4 + 1]);
      acc[4 * j4 + 2] = fmaf(wv.z, x, acc[4 * j4 + 2]);
      acc[4 * j4 + 3] = fmaf(wv.w, x, acc[4 * j4 + 3]);
    }
  }
}

struct PolArgs {
  int64_t n;
  int32_t obs_dim, act_dim, pi_h1, pi_h2, v_h1, v_h2;
  const float* obs;
  const float* mean;
  const float* std;         // nullptr: no standardisation
  float eps;
  const float* pi_w[3]; const float* pi_b[3];
  const float* v_w[3]; const float* v_b[3];
  const float* log_std;
  const float* packed;      // [pi_words + v_words] packed weights (k_pack_policy)
  uint64_t seed, counter;
  int64_t env_offset;       // global index of row 0: the action noise does not depend on the sharding
  float* act; float* val; float* logp; float* mu;
};

// shared layout (floats): norm_mean[D], norm_inv[D], then per net: W1t[D][H], b1[H], W2t[H][H], b2[H], W3t[H][O4], b3[O4],
// then hid[kHidMax][kPolBlock]
template <int H>
__device__ __forceinline__ void run_net(const float* __restrict__ sm_net, const float* __restrict__ obs_row,
                                        const float* __restrict__ nmean, const float* __restrict__ ninv, int D, int h1, int h2,
                                        bool tanh_act, float* __restrict__ hid, int tid, float (&out)[4]) {
  const float* w1 = sm_net;
  const float* b1 = w1 + D * H;
  const float* w2 = b1 + H;
  const float* b2 = w2 + H * H;
  const float* w3 = b2 + H;
  const float* b3 = w3 + H * 4;
  float acc[H];
  dense<H>(w1, b1, D, [&](int i) { return (__ldg(obs_row + i) - nmean[i]) * ninv[i]; }, acc);
#pragma unroll
  for (int j = 0; j < H; ++j) hid[j * kPolBlock + tid] = tanh_act ? fast_tanh(acc[j]) : fmaxf(acc[j], 0.0f);
  dense<H>(w2, b2, h1, [&](int i) { return hid[i * kPolBlock + tid]; }, acc);
  // every thread owns its hid column: no barrier needed between the read loop above and these writes
#pragma unroll
  for (int j = 0; j < H; ++j) hid[j * kPolBlock + tid] = tanh_act ? fast_tanh(acc[j]) : fmaxf(acc[j], 0.0f);
  dense<4>(w3, b3, h2, [&](int i) { return hid[i * kPolBlock + tid]; }, out);
}

// Packs torch nn.Linear weights ([out][in]) into the kernel's shared-memory image: per net
// W1t[D][H], b1[H], W2t[H][H], b2[H], W3t[H][4], b3[4], zero padded to H (52 or 64).
template <int HP, int HV>
__global__ void k_pack_policy(const PolArgs a, float* __restrict__ out) {
  const int D = a.obs_dim;
  const int pi_words = pdx::policy_net_words(D, HP);
  auto pack = [&](float* net, int H, const float* const* w, const float* const* b, int h1, int h2, int n_out) {
    float* w1 = net; float* b1 = w1 + D * H; float* w2 = b1 + H; float* b2 = w2 + H * H; float* w3 = b2 + H; float* b3 = w3 + H * 4;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int k = tid; k < D * H; k += nt) { const int i = k / H, j = k % H; w1[k] = j < h1 ? w[0][j * D + i] : 0.0f; }
    for (int k = tid; k < H; k += nt) { b1[k] = k < h1 ? b[0][k] : 0.0f; b2[k] = k < h2 ? b[1][k] : 0.0f; }
    for (int k = tid; k < H * H; k += nt) { const int i = k / H, j = k % H; w2[k] = (j < h2 && i < h1) ? w[1][j * h1 + i] : 0.0f; }
    for (int k = tid; k < H * 4; k += nt) { const int i = k / 4, j = k % 4; w3[k] = (j < n_out && i < h2) ? w[2][j * h2 + i] : 0.0f; }
    if (tid < 4) b3[tid] = tid < n_out ? b[2][tid] : 0.0f;
  };
  pack(out, HP, a.pi_w, a.pi_b, a.pi_h1, a.pi_h2, a.act_dim);
  pack(out + pi_words, HV, a.v_w, a.v_b, a.v_h1, a.v_h2, 1);
}

template <int HP, int HV>
__global__ void __launch_bounds__(kPolBlock) k_policy(const PolArgs a) {
#include "pdx_policy_body.cuh"
}

// A population's policy step: member m = blockIdx.y runs k_policy's body on its own slices -- obs / act / val / logp /
// mu [P][n][.], normaliser [P][D], log_std [P][act_dim], image [P][stride] -- and draws its noise at the global
// environment index env_offset + m n + i, so its outputs equal pdx_policy_step on its rows bit for bit
template <int HP, int HV>
__global__ void __launch_bounds__(kPolBlock) k_policy_members(const PolArgs args, int64_t stride) {
  const int64_t m = blockIdx.y, n = args.n;
  PolArgs a = args;
  a.obs = args.obs + m * n * args.obs_dim;
  if (args.std) { a.mean = args.mean + m * args.obs_dim; a.std = args.std + m * args.obs_dim; }
  a.log_std = args.log_std + m * args.act_dim;
  a.packed = args.packed + m * stride;
  a.env_offset = args.env_offset + m * n;
  a.act = args.act + m * n * 4; a.val = args.val + m * n; a.logp = args.logp + m * n;
  if (args.mu) a.mu = args.mu + m * n * 4;
#include "pdx_policy_body.cuh"
}

template <int HP, int HV>
int launch_policy_members(const PolArgs& a, int members, int64_t stride, int dev, cudaStream_t st) {
  const int D = a.obs_dim;
  const size_t words = 2 * ((D + 3) & ~3) + (size_t)pdx::policy_net_words(D, HP) + (size_t)pdx::policy_net_words(D, HV) +
                       (size_t)kHidMax * kPolBlock;
  const size_t smem = words * sizeof(float);
  if (smem > pdx::kMaxSmemBytes) return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: obs_dim too wide for the shared-memory plan");
  const int rc = pdx::cuda_error("pdx_policy_step_members (shared-memory opt-in)", pdx::opt_in_smem(k_policy_members<HP, HV>, dev, smem));
  if (rc) return rc;
  const dim3 grid((unsigned)((a.n + kPolBlock - 1) / kPolBlock), (unsigned)members);
  k_policy_members<HP, HV><<<grid, kPolBlock, smem, st>>>(a, stride);
  return pdx::cuda_error("pdx_policy_step_members", cudaGetLastError());
}

template <int HP, int HV>
int launch_policy(const PolArgs& a, int dev, cudaStream_t st) {
  const int D = a.obs_dim;
  const size_t words = 2 * ((D + 3) & ~3) + (size_t)pdx::policy_net_words(D, HP) + (size_t)pdx::policy_net_words(D, HV) +
                       (size_t)kHidMax * kPolBlock;
  const size_t smem = words * sizeof(float);
  if (a.n == 0) {                                     // pack only (pdx_evaluate stages the actor part of wider images)
    k_pack_policy<HP, HV><<<8, 256, 0, st>>>(a, const_cast<float*>(a.packed));
    return pdx::cuda_error("pdx_policy_pack", cudaGetLastError());
  }
  if (smem > pdx::kMaxSmemBytes) return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step: obs_dim too wide for the shared-memory plan");
  const int rc = pdx::cuda_error("pdx_policy_step (shared-memory opt-in)", pdx::opt_in_smem(k_policy<HP, HV>, dev, smem));
  if (rc) return rc;
  const unsigned grid = (unsigned)((a.n + kPolBlock - 1) / kPolBlock);
  k_policy<HP, HV><<<grid, kPolBlock, smem, st>>>(a);
  return pdx::cuda_error("pdx_policy_step", cudaGetLastError());
}

}  // namespace

static int policy_dispatch(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                           const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, uint64_t seed,
                           uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp, float* mu_out, void* stream);

extern "C" int64_t pdx_policy_pack_words(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v) {
  if (obs_dim <= 0 || !pi || !v) return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_pack_words: bad argument");
  return pdx::policy_net_words((int64_t)obs_dim, pdx::policy_actor_pad(pi->hidden[0], pi->hidden[1])) + pdx::policy_net_words((int64_t)obs_dim, 64);
}

extern "C" int pdx_policy_pack(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, float* packed, void* stream) {
  if (!packed) return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_pack: null buffer");
  return policy_dispatch(0, obs_dim, packed, nullptr, nullptr, 0.f, pi, v, packed, packed, 0, 0, 0, packed, packed, packed, nullptr, stream);
}

extern "C" int pdx_policy_step(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                               const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, uint64_t seed,
                               uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp, float* mu_out, void* stream) {
  if (n <= 0) return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step: n must be positive");
  return policy_dispatch(n, obs_dim, obs, mean, std, eps, pi, v, log_std, packed, seed, counter, env_offset, actions, values, logp, mu_out, stream);
}

static int policy_dispatch(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                           const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, uint64_t seed,
                           uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp, float* mu_out, void* stream) {
  if (n < 0 || obs_dim <= 0 || !obs || !pi || !v || !log_std || !packed || !actions || !values || !logp)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step: null buffer or bad size");
  if (pi->hidden[0] < 1 || pi->hidden[0] > kHidMax || pi->hidden[1] < 1 || pi->hidden[1] > kHidMax || pi->n_out < 1 || pi->n_out > 4)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step: actor must have two hidden layers of <= 64 units and <= 4 outputs");
  if (v->hidden[0] < 1 || v->hidden[0] > kHidMax || v->hidden[1] < 1 || v->hidden[1] > kHidMax || v->n_out != 1)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step: critic must have two hidden layers of <= 64 units and one output");
  int dev = 0;
  const int rc = pdx::select_device_of(obs, &dev);
  if (rc) return rc;
  PolArgs a;
  a.n = n; a.obs_dim = obs_dim; a.act_dim = pi->n_out;
  a.pi_h1 = pi->hidden[0]; a.pi_h2 = pi->hidden[1]; a.v_h1 = v->hidden[0]; a.v_h2 = v->hidden[1];
  a.obs = obs; a.mean = mean; a.std = std; a.eps = eps;
  for (int k = 0; k < 3; ++k) { a.pi_w[k] = pi->weight[k]; a.pi_b[k] = pi->bias[k]; a.v_w[k] = v->weight[k]; a.v_b[k] = v->bias[k]; }
  a.log_std = log_std; a.packed = packed; a.seed = seed; a.counter = counter; a.env_offset = env_offset;
  a.act = actions; a.val = values; a.logp = logp; a.mu = mu_out;
  const cudaStream_t st = (cudaStream_t)stream;
  return pdx::policy_actor_pad(a.pi_h1, a.pi_h2) == 52 ? launch_policy<52, 64>(a, dev, st) : launch_policy<64, 64>(a, dev, st);
}

extern "C" int pdx_policy_step_members(int32_t members, int64_t n, int32_t obs_dim, const float* obs, const float* mean,
                                       const float* std, float eps, const PdxMlp* pi, const PdxMlp* v,
                                       const float* log_std, const float* packed, int64_t stride, uint64_t seed,
                                       uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp,
                                       float* mu_out, void* stream) {
  if (members < 1 || members > 65535 || n <= 0 || obs_dim <= 0 || obs_dim > 384)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: members in [1, 65535], n >= 1 and obs_dim in [1, 384]");
  if (!obs || !pi || !v || !log_std || !packed || !actions || !values || !logp || (!mean) != (!std))
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: null buffer (mean and std: both or neither)");
  if (pi->hidden[0] < 1 || pi->hidden[0] > kHidMax || pi->hidden[1] < 1 || pi->hidden[1] > kHidMax || pi->n_out < 1 || pi->n_out > 4)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: actor must have two hidden layers of <= 64 units and <= 4 outputs");
  if (v->hidden[0] < 1 || v->hidden[0] > kHidMax || v->hidden[1] < 1 || v->hidden[1] > kHidMax || v->n_out != 1)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: critic must have two hidden layers of <= 64 units and one output");
  const int HP = pdx::policy_actor_pad(pi->hidden[0], pi->hidden[1]);
  if (stride < pdx::policy_net_words((int64_t)obs_dim, HP) + pdx::policy_net_words((int64_t)obs_dim, 64) || stride % 4)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: stride must be a multiple of 4 and >= pdx_policy_pack_words()");
  const size_t words = 2 * ((obs_dim + 3) & ~3) + (size_t)pdx::policy_net_words(obs_dim, HP) +
                       (size_t)pdx::policy_net_words(obs_dim, 64) + (size_t)kHidMax * kPolBlock;
  if (words * sizeof(float) > pdx::kMaxSmemBytes)
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_members: obs_dim too wide for the shared-memory plan");
  int dev = 0;
  const int rc = pdx::select_device_of(obs, &dev);
  if (rc) return rc;
  PolArgs a;
  a.n = n; a.obs_dim = obs_dim; a.act_dim = pi->n_out;
  a.pi_h1 = pi->hidden[0]; a.pi_h2 = pi->hidden[1]; a.v_h1 = v->hidden[0]; a.v_h2 = v->hidden[1];
  a.obs = obs; a.mean = mean; a.std = std; a.eps = eps;
  for (int k = 0; k < 3; ++k) { a.pi_w[k] = pi->weight[k]; a.pi_b[k] = pi->bias[k]; a.v_w[k] = v->weight[k]; a.v_b[k] = v->bias[k]; }
  a.log_std = log_std; a.packed = packed; a.seed = seed; a.counter = counter; a.env_offset = env_offset;
  a.act = actions; a.val = values; a.logp = logp; a.mu = mu_out;
  const cudaStream_t st = (cudaStream_t)stream;
  return HP == 52 ? launch_policy_members<52, 64>(a, members, stride, dev, st) : launch_policy_members<64, 64>(a, members, stride, dev, st);
}
