// pdx_ppo_pi_grad / pdx_ppo_v_grad: the losses of PPO's update (algs/ppo/ppo.py:22-40, algs/iwpg/iwpg.py:446-485)
// and their exact gradients with respect to every nn.Linear weight and bias of one network, on the CUDA cores in float32.
// pdx_ppo_pi_fvp: NPG / TRPO's Fisher-vector product (algs/npg/npg.py Fvp) on the same plan, with a tangent pass
// along the direction between the forward and the backward pass (k_ppo_fvp).
//
// Design
//   * persistent grid, fixed assignment of sample tiles to CTAs (tile t -> CTA t mod G); one thread per sample of a
//     tile of S samples (S = blockDim = 128, fewer for wide observations so that the plan fits shared memory).
//   * the block stages the network once from the torch tensors ([out][in] row-major): W1t[D+1][H] and W2t[h1+1][H]
//     transposed for the forward pass with the bias as an extra input row, W2[H][H] as is for the backward pass,
//     W3t[H][4].  H = 52 or 64 (zero padding).  Every activation tile carries a constant-1 column after its last unit,
//     so the bias is just one more input of the forward pass and one more column of the weight-gradient product.
//   * per tile, each thread runs the forward pass and the backward data pass of its sample (accumulators in
//     registers, weights read as 128-bit shared-memory broadcasts as in k_policy) and writes X, a1, a2, d1, d2, d3
//     into shared-memory tiles.  The block then forms G_l = d_l^T [a_{l-1}, 1] for the three layers as one list of
//     4 x 4 register patches (a patch sums its tile in float32, in sample order) and adds each patch into the
//     CTA's float64 partial in `scratch`; a patch always belongs to the same thread of the same CTA.
//   * k_ppo_reduce sums the G partials of every entry in CTA order in float64, divides by n and writes the float32
//     gradients into the caller's tensors, and the loss (and KL) as float32 device scalars.
//   Hence the results are bit-identical from run to run for the same device, inputs and scratch size.
//
// Arithmetic per sample (D inputs, h1 / h2 hidden units, O outputs): forward D h1 + h1 h2 + O h2 FMAs, backward data
// O h2 + h1 h2, weight gradients D h1 + h1 h2 + O h2 (biases aside).  This unit is built without -use_fast_math:
// expf and tanhf are the accurate ones.
#include <cmath>

#include "pdx_host.h"
#include "pdx_layout.h"

namespace pdx {
namespace {

constexpr int kPpoMaxBlock = 128;
constexpr int kPpoMaxObs = 384;               // history 16 of the widest task: 16 * (20 + 4)

__host__ __device__ constexpr int round4(int x) { return (x + 3) & ~3; }
// row stride (floats) of a tile holding `cols` columns: a multiple of 4 whose float4 count is odd, so that 32 threads
// reading 16 bytes each of their own rows hit every bank once per 8 threads
__host__ __device__ constexpr int tile_stride(int cols) { return (round4(cols) / 4) % 2 ? round4(cols) : round4(cols) + 4; }
__host__ __device__ constexpr int act_stride(int H) { return tile_stride(H + 1); }

// gradient entries of one network (G1 [h1][D+1], G2 [h2][h1+1], G3 [O][h2+1]) plus the loss and KL sums
__host__ __device__ inline int ppo_entries(int D, int h1, int h2, int O) { return h1 * (D + 1) + h2 * (h1 + 1) + O * (h2 + 1) + 2; }

// shared-memory plan (floats): W1t[round4(D+1)][H], W2t[H+4][H], W2[H][H], W3t[H][4], b3[4];
// tiles X[S][tile_stride(D+1)], A1, A2, D1, D2 [S][act_stride(H)], D3[S][4]; the final reduction's S doubles.
// The Fisher-vector product (fvp) adds dW3t[H][4], db3[4], gives W2 H + 4 rows (it holds dW2t during the tangent
// pass, W1t holds dW1t) and needs no loss reduction.
inline size_t ppo_smem_bytes(int S, int D, int H, bool fvp = false) {
  const size_t w = (size_t)round4(D + 1) * H + (size_t)(H + 4) * H + (size_t)(fvp ? H + 4 : H) * H + (fvp ? 8 : 4) * H +
                   (fvp ? 8 : 4);
  const size_t t = (size_t)S * tile_stride(D + 1) + 4 * (size_t)S * act_stride(H) + 4 * (size_t)S + (fvp ? 0 : 2 * (size_t)S);
  return (w + t) * sizeof(float);
}

struct PpoArgs {
  int64_t n, ntiles;
  int32_t D, h1, h2, O, E2;                   // E2 = ppo_entries
  const float* obs; const int64_t* index;
  const float* act; const float* adv; const float* logp_old; const float* target_v;
  const float* w[3]; const float* b[3];
  const float* log_std;
  float lo, hi;                               // 1 - clip_ratio, 1 + clip_ratio
  float* mu; const float* mu_ref;
  double* part;                               // [G][E2]
  const float* dw[3]; const float* db[3];     // fvp: the direction, shaped like the network
};

// what one k_ppo-plan launch computes
enum PpoKind { kCritic, kClipped, kUnclipped, kFvp };

// acc[j] += sum_{i < nin4} W[i][j] in[i] for the H outputs (W row stride H), inputs in order
template <int H>
__device__ __forceinline__ void dense_add(const float* __restrict__ W, int nin4, const float* __restrict__ in, float (&acc)[H]) {
  for (int i = 0; i < nin4; i += 4) {
    const float4 x4 = *reinterpret_cast<const float4*>(in + i);
    const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4* row = reinterpret_cast<const float4*>(W + (i + q) * H);
#pragma unroll
      for (int j4 = 0; j4 < H / 4; ++j4) {
        const float4 wv = row[j4];
        acc[4 * j4 + 0] = fmaf(wv.x, xs[q], acc[4 * j4 + 0]);
        acc[4 * j4 + 1] = fmaf(wv.y, xs[q], acc[4 * j4 + 1]);
        acc[4 * j4 + 2] = fmaf(wv.z, xs[q], acc[4 * j4 + 2]);
        acc[4 * j4 + 3] = fmaf(wv.w, xs[q], acc[4 * j4 + 3]);
      }
    }
  }
}

template <int H>
__device__ __forceinline__ void dense(const float* __restrict__ W, int nin4, const float* __restrict__ in, float (&acc)[H]) {
#pragma unroll
  for (int j = 0; j < H; ++j) acc[j] = 0.0f;
  dense_add<H>(W, nin4, in, acc);
}

// dst[i][j] = [W | b]^T of an [nout][nin] layer with the bias as input row nin, zero padded to `rows` x H
template <int H>
__device__ __forceinline__ void stage_t(float* dst, int rows, const float* W, const float* b, int nin, int nout) {
  for (int k = threadIdx.x; k < rows * H; k += blockDim.x) {
    const int i = k / H, j = k % H;
    dst[k] = j < nout ? (i < nin ? W[j * nin + i] : i == nin ? b[j] : 0.0f) : 0.0f;
  }
}

// dst[j][i] = W[j][i] of an [nout][nin] layer, zero padded to H x H
template <int H>
__device__ __forceinline__ void stage_w(float* dst, const float* W, int nin, int nout) {
  for (int k = threadIdx.x; k < H * H; k += blockDim.x) {
    const int j = k / H, i = k % H;
    dst[k] = (j < nout && i < nin) ? W[j * nin + i] : 0.0f;
  }
}

template <bool ACTOR>
__device__ __forceinline__ float act_fn(float z) { return ACTOR ? (z > 0.0f ? z : 0.0f) : tanhf(z); }
// derivative from the activation's output: relu' = 1 only for z > 0 (torch threshold_backward), tanh' = 1 - a^2
template <bool ACTOR>
__device__ __forceinline__ float act_grad(float a) { return ACTOR ? (a > 0.0f ? 1.0f : 0.0f) : 1.0f - a * a; }

template <int KIND, bool GRAD, int H>
__device__ __forceinline__ void ppo_body(const PpoArgs& a) {
  constexpr bool ACTOR = KIND != kCritic, FVP = KIND == kFvp;
  constexpr int AS = act_stride(H);
  const int S = blockDim.x, tid = threadIdx.x;
  const int D = a.D, h1 = a.h1, h2 = a.h2, O = a.O;
  const int D1 = round4(D + 1), XS = tile_stride(D + 1);
  extern __shared__ __align__(16) float ppo_sm[];
  float* w1t = ppo_sm;                        // [D1][H]
  float* w2t = w1t + D1 * H;                  // [H + 4][H]
  float* w2b = w2t + (H + 4) * H;             // [H][H] (fvp: [H + 4][H])
  float* w3t = w2b + (FVP ? H + 4 : H) * H;   // [H][4]
  float* b3 = w3t + 4 * H;                    // [4]
  float* dw3t = b3 + 4;                       // fvp: [H][4]
  float* db3 = dw3t + 4 * H;                  // fvp: [4]
  float* X = FVP ? db3 + 4 : b3 + 4;          // [S][XS]
  float* A1 = X + S * XS;
  float* A2 = A1 + S * AS;
  float* D1t = A2 + S * AS;
  float* D2t = D1t + S * AS;
  float* D3t = D2t + S * AS;                  // [S][4]
  double* red = reinterpret_cast<double*>(D3t + 4 * S);

  for (int k = tid; k < D1 * H; k += S) {
    const int i = k / H, j = k % H;
    w1t[k] = j < h1 ? (i < D ? a.w[0][j * D + i] : i == D ? a.b[0][j] : 0.0f) : 0.0f;
  }
  for (int k = tid; k < (H + 4) * H; k += S) {
    const int i = k / H, j = k % H;
    w2t[k] = j < h2 ? (i < h1 ? a.w[1][j * h1 + i] : i == h1 ? a.b[1][j] : 0.0f) : 0.0f;
  }
  for (int k = tid; k < H * H; k += S) {
    const int j = k / H, i = k % H;
    w2b[k] = (j < h2 && i < h1) ? a.w[1][j * h1 + i] : 0.0f;
  }
  for (int k = tid; k < 4 * H; k += S) {
    const int j = k / 4, o = k % 4;
    w3t[k] = (j < h2 && o < O) ? a.w[2][o * h2 + j] : 0.0f;
  }
  if (tid < 4) b3[tid] = tid < O ? a.b[2][tid] : 0.0f;
  if (FVP) {
    for (int k = tid; k < 4 * H; k += S) {
      const int j = k / 4, o = k % 4;
      dw3t[k] = j < h2 ? a.dw[2][o * h2 + j] : 0.0f;
    }
    if (tid < 4) db3[tid] = a.db[2][tid];
  }
  float ls[4] = {0.f, 0.f, 0.f, 0.f}, sd[4] = {1.f, 1.f, 1.f, 1.f};
  if (ACTOR) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { ls[k] = a.log_std[k]; sd[k] = expf(ls[k]); }
  }

  const int P1 = ((h1 + 3) / 4) * ((D + 4) / 4), P2 = ((h2 + 3) / 4) * ((h1 + 4) / 4), P3 = ((h2 + 4) / 4);
  double* part = a.part + (int64_t)blockIdx.x * a.E2;
  double lsum = 0.0, ksum = 0.0;
  float* xr = X + tid * XS; float* a1r = A1 + tid * AS; float* a2r = A2 + tid * AS;
  float* d1r = D1t + tid * AS; float* d2r = D2t + tid * AS; float* d3r = D3t + 4 * tid;

  for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int64_t base = tile * S;
    __syncthreads();                          // the previous tile's readers are done with X (and the weights staged)
    if (FVP && tile != blockIdx.x) stage_t<H>(w1t, D1, a.w[0], a.b[0], D, h1);    // dW1t during the tangent pass
    for (int k = tid; k < S * XS; k += S) {
      const int s = k / XS, c = k - s * XS;
      const int64_t i = base + s;
      float v = 0.0f;
      if (i < a.n) {
        const int64_t row = a.index ? a.index[i] : i;
        v = c < D ? a.obs[row * D + c] : c == D ? 1.0f : 0.0f;
      }
      X[k] = v;
    }
    __syncthreads();
    // ---- this thread's sample: forward pass
    const int64_t i = base + tid;
    const bool valid = i < a.n;
    const int64_t row = valid ? (a.index ? a.index[i] : i) : 0;
    float acc[H];
    dense<H>(w1t, D1, xr, acc);
#pragma unroll
    for (int j4 = 0; j4 < AS / 4; ++j4) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = 4 * j4 + q < H ? act_fn<ACTOR>(acc[4 * j4 + q]) : 0.0f;
      *reinterpret_cast<float4*>(a1r + 4 * j4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    a1r[h1] = 1.0f;                           // unit h1 is padding (or past H): the bias input of layer 2
    dense<H>(w2t, round4(h1 + 1), a1r, acc);
    float out[4] = {b3[0], b3[1], b3[2], b3[3]};
#pragma unroll
    for (int j4 = 0; j4 < AS / 4; ++j4) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = 4 * j4 + q;
        v[q] = j < H ? act_fn<ACTOR>(acc[j]) : 0.0f;
        if (j < H) {
          const float4 wv = reinterpret_cast<const float4*>(w3t)[j];
          out[0] = fmaf(wv.x, v[q], out[0]); out[1] = fmaf(wv.y, v[q], out[1]);
          out[2] = fmaf(wv.z, v[q], out[2]); out[3] = fmaf(wv.w, v[q], out[3]);
        }
      }
      *reinterpret_cast<float4*>(a2r + 4 * j4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    a2r[h2] = 1.0f;
    // ---- loss term and d loss / d output (without the 1 / n of the mean, applied in float64 by k_ppo_reduce)
    float d3[4] = {0.f, 0.f, 0.f, 0.f};
    if (FVP) {
      // ---- tangent pass along the direction: u = J dir, J = d mu / d theta of this sample; d3 = u / std^2
      __syncthreads();                        // every thread is done with W1t and W2
      stage_t<H>(w1t, D1, a.dw[0], a.db[0], D, h1);
      stage_t<H>(w2b, H + 4, a.dw[1], a.db[1], h1, h2);
      __syncthreads();
      dense<H>(w1t, D1, xr, acc);            // dz1 = dW1 [x, 1]
#pragma unroll
      for (int j4 = 0; j4 < AS / 4; ++j4) {  // da1 = dz1 relu'(z1) into the D1 row (the backward pass overwrites it);
        float v[4];                           // entry h1 is 0, the bias input of [da1, 0]
        const float4 av = *reinterpret_cast<const float4*>(a1r + 4 * j4);
        const float as[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = 4 * j4 + q < H ? acc[4 * j4 + q] * act_grad<true>(as[q]) : 0.0f;
        *reinterpret_cast<float4*>(d1r + 4 * j4) = make_float4(v[0], v[1], v[2], v[3]);
      }
      dense<H>(w2b, round4(h1 + 1), a1r, acc);        // dz2 = dW2 [a1, 1] + W2 [da1, 0]
      dense_add<H>(w2t, round4(h1 + 1), d1r, acc);
      float u[4] = {db3[0], db3[1], db3[2], db3[3]};  // u = dW3 [a2, 1] + W3 (dz2 relu'(z2))
#pragma unroll
      for (int j4 = 0; j4 < H / 4; ++j4) {
        const float4 av = *reinterpret_cast<const float4*>(a2r + 4 * j4);
        const float as[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int j = 4 * j4 + q;
          const float da2 = acc[j] * act_grad<true>(as[q]);
          const float4 dv = reinterpret_cast<const float4*>(dw3t)[j], wv = reinterpret_cast<const float4*>(w3t)[j];
          u[0] = fmaf(wv.x, da2, fmaf(dv.x, as[q], u[0])); u[1] = fmaf(wv.y, da2, fmaf(dv.y, as[q], u[1]));
          u[2] = fmaf(wv.z, da2, fmaf(dv.z, as[q], u[2])); u[3] = fmaf(wv.w, da2, fmaf(dv.w, as[q], u[3]));
        }
      }
      if (valid) {
#pragma unroll
        for (int k = 0; k < 4; ++k) d3[k] = u[k] / (sd[k] * sd[k]);
      }
      __syncthreads();                        // every thread is done with dW2t: W2 back for the backward pass
      stage_w<H>(w2b, a.w[1], h1, h2);
      __syncthreads();
    } else if (valid) {
      if (ACTOR) {
        float z[4], lp = 0.0f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          z[k] = (a.act[row * 4 + k] - out[k]) / sd[k];
          lp += -0.5f * z[k] * z[k] - ls[k] - 0.9189385332046727f;
        }
        const float A = a.adv[row];
        const float r = expf(lp - a.logp_old[row]);
        const float s1 = r * A;
        float g;
        if (KIND == kUnclipped) {             // -(r A).mean(): a non-finite ratio reaches the loss, as in torch
          lsum -= (double)s1;
          g = -s1;
        } else {
          const float s2 = fminf(fmaxf(r, a.lo), a.hi) * A;
          lsum -= (double)fminf(s1, s2);
          // torch: minimum passes the gradient to r A where r A <= clip(r) A (a tie inside the clip range is a tie of
          // r A with itself); clamp passes nothing outside [lo, hi].  d logp / d mu = (a - mu) / std^2
          g = s1 <= s2 ? -s1 : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) d3[k] = g * z[k] / sd[k];
        if (a.mu) {
#pragma unroll
          for (int k = 0; k < 4; ++k) a.mu[i * 4 + k] = out[k];
        }
        if (a.mu_ref) {
          float kl = 0.0f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float d = a.mu_ref[i * 4 + k] - out[k];
            kl += d * d / (2.0f * sd[k] * sd[k]);
          }
          ksum += (double)kl;
        }
      } else {
        const float d = out[0] - a.target_v[row];
        lsum += (double)(d * d);
        d3[0] = 2.0f * d;
      }
    }
    if (GRAD) {
      // ---- backward data pass: d2 = (W3^T d3) f'(a2), d1 = (W2^T d2) f'(a1)
      *reinterpret_cast<float4*>(d3r) = make_float4(d3[0], d3[1], d3[2], d3[3]);
#pragma unroll
      for (int j4 = 0; j4 < H / 4; ++j4) {
        const float4 av = *reinterpret_cast<const float4*>(a2r + 4 * j4);
        const float as[4] = {av.x, av.y, av.z, av.w};
        float v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 wv = reinterpret_cast<const float4*>(w3t)[4 * j4 + q];
          const float s = fmaf(wv.w, d3[3], fmaf(wv.z, d3[2], fmaf(wv.y, d3[1], wv.x * d3[0])));
          v[q] = s * act_grad<ACTOR>(as[q]);
        }
        *reinterpret_cast<float4*>(d2r + 4 * j4) = make_float4(v[0], v[1], v[2], v[3]);
      }
      dense<H>(w2b, round4(h2), d2r, acc);
#pragma unroll
      for (int j4 = 0; j4 < H / 4; ++j4) {
        const float4 av = *reinterpret_cast<const float4*>(a1r + 4 * j4);
        *reinterpret_cast<float4*>(d1r + 4 * j4) =
            make_float4(acc[4 * j4 + 0] * act_grad<ACTOR>(av.x), acc[4 * j4 + 1] * act_grad<ACTOR>(av.y),
                        acc[4 * j4 + 2] * act_grad<ACTOR>(av.z), acc[4 * j4 + 3] * act_grad<ACTOR>(av.w));
      }
      __syncthreads();
      // ---- weight gradients of the tile: G1 = d1^T [X, 1], G2 = d2^T [a1, 1], G3 = d3^T [a2, 1] in 4 x 4 patches
      const bool first = tile == blockIdx.x;
      for (int p = tid; p < P1 + P2 + P3; p += S) {
        const float* dl; const float* al; int ldd, lda, R, C, q; double* o;
        if (p < P1) { dl = D1t; ldd = AS; al = X; lda = XS; R = h1; C = D + 1; q = p; o = part; }
        else if (p < P1 + P2) { dl = D2t; ldd = AS; al = A1; lda = AS; R = h2; C = h1 + 1; q = p - P1; o = part + h1 * (D + 1); }
        else { dl = D3t; ldd = 4; al = A2; lda = AS; R = O; C = h2 + 1; q = p - P1 - P2; o = part + h1 * (D + 1) + h2 * (h1 + 1); }
        const int CP = (C + 3) / 4, r0 = 4 * (q / CP), c0 = 4 * (q % CP);
        float g[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) g[r][c] = 0.0f;
#pragma unroll 4
        for (int s = 0; s < S; ++s) {
          const float4 dv = *reinterpret_cast<const float4*>(dl + s * ldd + r0);
          const float4 xv = *reinterpret_cast<const float4*>(al + s * lda + c0);
          const float ds[4] = {dv.x, dv.y, dv.z, dv.w}, xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
          for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) g[r][c] = fmaf(ds[r], xs[c], g[r][c]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (r0 + r < R && c0 + c < C) {
              double* e = o + (r0 + r) * C + c0 + c;
              *e = first ? (double)g[r][c] : *e + (double)g[r][c];
            }
      }
    }
  }
  if (FVP) return;                            // no loss: the reduction's entries E2 - 2, E2 - 1 are not written
  // ---- loss and KL sums of this CTA, in thread order
  __syncthreads();
  red[tid] = lsum;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int k = 0; k < S; ++k) s += red[k];
    part[a.E2 - 2] = s;
  }
  __syncthreads();
  red[tid] = ksum;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int k = 0; k < S; ++k) s += red[k];
    part[a.E2 - 1] = s;
  }
}

template <bool ACTOR, bool GRAD, int H>
__global__ void __launch_bounds__(kPpoMaxBlock) k_ppo(const PpoArgs a) { ppo_body<ACTOR ? kClipped : kCritic, GRAD, H>(a); }

template <bool GRAD, int H>
__global__ void __launch_bounds__(kPpoMaxBlock) k_ppo_unclipped(const PpoArgs a) { ppo_body<kUnclipped, GRAD, H>(a); }

// J^T diag(std^-2) J dir summed over the samples (J = d mu / d theta): the tangent pass gives u = J dir, the backward
// pass and the weight-gradient patches of the actor's gradient turn d3 = u / std^2 into J^T d3
template <int H>
__global__ void __launch_bounds__(kPpoMaxBlock) k_ppo_fvp(const PpoArgs a) { ppo_body<kFvp, true, H>(a); }

struct ReduceArgs {
  int32_t G, D, h1, h2, O, E2;
  double inv_n;
  const double* part;
  float* gw[3]; float* gb[3];                 // NULL: forward only
  float* loss; float* kl;
};

// entry e of every CTA's partial summed in CTA order, / n, into the gradient tensors ([out][in] + bias) / loss / kl
__global__ void k_ppo_reduce(const ReduceArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E2 || (!a.gw[0] && e < a.E2 - 2)) return;
  double s = 0.0;
  for (int g = 0; g < a.G; ++g) s += a.part[(int64_t)g * a.E2 + e];
  const float v = (float)(s * a.inv_n);
  if (e == a.E2 - 2) { *a.loss = v; return; }
  if (e == a.E2 - 1) { if (a.kl) *a.kl = v; return; }
  int l = 0, in = a.D, k = e;
  if (k >= a.h1 * (a.D + 1)) { k -= a.h1 * (a.D + 1); l = 1; in = a.h1;
    if (k >= a.h2 * (a.h1 + 1)) { k -= a.h2 * (a.h1 + 1); l = 2; in = a.h2; } }
  const int r = k / (in + 1), c = k % (in + 1);
  if (c < in) (l == 0 ? a.gw[0] : l == 1 ? a.gw[1] : a.gw[2])[r * in + c] = v;
  else (l == 0 ? a.gb[0] : l == 1 ? a.gb[1] : a.gb[2])[r] = v;
}

struct FvpReduceArgs {
  int32_t G, D, h1, h2, E2;
  double scale_n, damping;                    // scale / n
  const double* part;
  const float* dw[3]; const float* db[3];     // the direction
  float* gw[3]; float* gb[3];
};

// k_ppo_reduce for the Fisher-vector product: out = scale / n * (sum of the CTA partials in CTA order) + damping * dir,
// in float64, rounded once
__global__ void k_ppo_fvp_reduce(const FvpReduceArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E2 - 2) return;
  double s = 0.0;
  for (int g = 0; g < a.G; ++g) s += a.part[(int64_t)g * a.E2 + e];
  int l = 0, in = a.D, k = e;
  if (k >= a.h1 * (a.D + 1)) { k -= a.h1 * (a.D + 1); l = 1; in = a.h1;
    if (k >= a.h2 * (a.h1 + 1)) { k -= a.h2 * (a.h1 + 1); l = 2; in = a.h2; } }
  const int r = k / (in + 1), c = k % (in + 1);
  const float* d = c < in ? a.dw[l] + r * in + c : a.db[l] + r;
  float* o = c < in ? a.gw[l] + r * in + c : a.gb[l] + r;
  *o = (float)(s * a.scale_n + a.damping * (double)*d);
}

bool mlp_ok(const PdxMlp* m, int n_out) {
  if (!m || m->hidden[0] < 1 || m->hidden[0] > 64 || m->hidden[1] < 1 || m->hidden[1] > 64 || m->n_out != n_out) return false;
  for (int k = 0; k < 3; ++k)
    if (!m->weight[k] || !m->bias[k]) return false;
  return true;
}

bool grad_ok(const PdxMlpGrad* g) {
  for (int k = 0; k < 3; ++k)
    if (!g->weight[k] || !g->bias[k]) return false;
  return true;
}

// tile size: the largest of 128, 64, 32 whose shared-memory plan fits
int ppo_tile(int D, int H, bool fvp) {
  for (int S = kPpoMaxBlock; S >= 32; S /= 2)
    if (ppo_smem_bytes(S, D, H, fvp) <= kMaxSmemBytes) return S;
  return 0;
}

template <typename K>
cudaError_t launch_ppo(K kernel, const PpoArgs& a, int S, size_t smem, int G, int dev, cudaStream_t st) {
  const cudaError_t e = opt_in_smem(kernel, dev, smem);
  if (e != cudaSuccess) return e;
  kernel<<<G, S, smem, st>>>(a);
  return cudaGetLastError();
}

template <int H>
cudaError_t launch_kind(int kind, bool grad, const PpoArgs& a, int S, size_t smem, int G, int dev, cudaStream_t st) {
  switch (kind) {
    case kCritic: return launch_ppo(k_ppo<false, true, H>, a, S, smem, G, dev, st);
    case kClipped: return launch_ppo(grad ? k_ppo<true, true, H> : k_ppo<true, false, H>, a, S, smem, G, dev, st);
    case kUnclipped: return launch_ppo(grad ? k_ppo_unclipped<true, H> : k_ppo_unclipped<false, H>, a, S, smem, G, dev, st);
    default: return launch_ppo(k_ppo_fvp<H>, a, S, smem, G, dev, st);
  }
}

// one launch of the k_ppo plan and its reduction.  kFvp: `grad` receives the product, dir / scale / damping are used
int ppo_run(const char* what, int kind, const PdxPpoBatch* b, const PdxMlp* net, const float* log_std, float clip_ratio,
            const PdxMlpGrad* grad, float* loss, float* mu, const float* mu_ref, float* kl, const PdxMlp* dir,
            float scale, float damping, void* scratch, int64_t scratch_bytes, void* stream) {
  const bool actor = kind != kCritic, fvp = kind == kFvp;
  const int D = b->obs_dim, h1 = net->hidden[0], h2 = net->hidden[1], O = actor ? 4 : 1;
  const int H = (h1 <= 52 && h2 <= 52) ? 52 : 64;
  const int S = ppo_tile(D, H, fvp);
  if (S == 0) return set_error(PDX_ERR_INVALID, "pdx_ppo: obs_dim too wide for the shared-memory plan");
  const int E2 = ppo_entries(D, h1, h2, O);
  const int64_t per_cta = (int64_t)E2 * sizeof(double);
  if (!scratch || scratch_bytes < per_cta)
    return set_error(PDX_ERR_INVALID, "pdx_ppo: scratch of pdx_ppo_scratch_bytes() bytes required");
  int dev = 0;
  int rc = select_device_of(b->obs, &dev);
  if (rc) return rc;
  int sms = 148;
  rc = cuda_error(what, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (rc) return rc;
  PpoArgs a;
  a.n = b->n; a.ntiles = (b->n + S - 1) / S;
  a.D = D; a.h1 = h1; a.h2 = h2; a.O = O; a.E2 = E2;
  a.obs = b->obs; a.index = b->index; a.act = b->act; a.adv = b->adv; a.logp_old = b->logp_old; a.target_v = b->target_v;
  for (int k = 0; k < 3; ++k) { a.w[k] = net->weight[k]; a.b[k] = net->bias[k]; }
  a.log_std = log_std;
  a.lo = (float)(1.0 - (double)clip_ratio); a.hi = (float)(1.0 + (double)clip_ratio);
  a.mu = mu; a.mu_ref = mu_ref;
  a.part = static_cast<double*>(scratch);
  for (int k = 0; k < 3; ++k) { a.dw[k] = fvp ? dir->weight[k] : nullptr; a.db[k] = fvp ? dir->bias[k] : nullptr; }
  int64_t G = a.ntiles < sms ? a.ntiles : sms;
  if (G > scratch_bytes / per_cta) G = scratch_bytes / per_cta;
  const cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = ppo_smem_bytes(S, D, H, fvp);
  const cudaError_t e = H == 52 ? launch_kind<52>(kind, grad != nullptr, a, S, smem, (int)G, dev, st)
                                : launch_kind<64>(kind, grad != nullptr, a, S, smem, (int)G, dev, st);
  if (e != cudaSuccess) return cuda_error(what, e);
  if (fvp) {
    FvpReduceArgs r;
    r.G = (int)G; r.D = D; r.h1 = h1; r.h2 = h2; r.E2 = E2; r.part = a.part;
    r.scale_n = (double)scale / (double)b->n; r.damping = damping;
    for (int k = 0; k < 3; ++k) { r.dw[k] = dir->weight[k]; r.db[k] = dir->bias[k]; r.gw[k] = grad->weight[k]; r.gb[k] = grad->bias[k]; }
    k_ppo_fvp_reduce<<<(E2 + 255) / 256, 256, 0, st>>>(r);
    return cuda_error(what, cudaGetLastError());
  }
  ReduceArgs r;
  r.G = (int)G; r.D = D; r.h1 = h1; r.h2 = h2; r.O = O; r.E2 = E2; r.inv_n = 1.0 / (double)b->n; r.part = a.part;
  for (int k = 0; k < 3; ++k) { r.gw[k] = grad ? grad->weight[k] : nullptr; r.gb[k] = grad ? grad->bias[k] : nullptr; }
  r.loss = loss; r.kl = kl;
  k_ppo_reduce<<<(E2 + 255) / 256, 256, 0, st>>>(r);
  return cuda_error(what, cudaGetLastError());
}

bool batch_ok(const PdxPpoBatch* b) {
  return b && b->n >= 1 && b->obs_dim >= 1 && b->obs_dim <= kPpoMaxObs && b->obs;
}

}  // namespace
}  // namespace pdx

extern "C" int64_t pdx_ppo_scratch_bytes(int32_t device, int32_t obs_dim, const PdxMlp* net) {
  using namespace pdx;
  if (obs_dim < 1 || obs_dim > kPpoMaxObs || !net || net->hidden[0] < 1 || net->hidden[0] > 64 || net->hidden[1] < 1 ||
      net->hidden[1] > 64 || (net->n_out != 1 && net->n_out != 4))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_scratch_bytes: bad argument");
  int n = 0;
  const int rc = count_devices(&n);
  if (rc) return rc;
  if (device < 0 || device >= n) return set_error(PDX_ERR_INVALID, "bad device ordinal");
  int sms = 0;
  const int e = cuda_error("pdx_ppo_scratch_bytes", cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (e) return e;
  return (int64_t)sms * ppo_entries(obs_dim, net->hidden[0], net->hidden[1], net->n_out) * (int64_t)sizeof(double);
}

extern "C" int pdx_ppo_pi_grad(const PdxPpoBatch* batch, const PdxMlp* pi, const float* log_std, float clip_ratio,
                               const PdxMlpGrad* grad, float* loss, float* mu, const float* mu_ref, float* kl,
                               void* scratch, int64_t scratch_bytes, void* stream) {
  using namespace pdx;
  if (!batch_ok(batch) || !batch->act || !batch->adv || !batch->logp_old)
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_grad: batch needs n >= 1, 1 <= obs_dim <= 384, obs, act, adv and logp_old");
  if (!mlp_ok(pi, 4) || !log_std)
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_grad: actor must have two hidden layers of <= 64 units, 4 outputs and log_std");
  const bool unclipped = clip_ratio == INFINITY;
  if (!(clip_ratio >= 0.0f && (clip_ratio < 1e30f || unclipped)))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_grad: clip_ratio must be >= 0 (finite, or +inf for no clip)");
  if (!loss || (grad && !grad_ok(grad)) || (!mu_ref) != (!kl))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_grad: loss is required, a gradient with all six tensors, mu_ref and kl both or neither");
  return ppo_run("pdx_ppo_pi_grad", unclipped ? kUnclipped : kClipped, batch, pi, log_std, clip_ratio, grad, loss, mu, mu_ref,
                 kl, nullptr, 0.0f, 0.0f, scratch, scratch_bytes, stream);
}

extern "C" int pdx_ppo_pi_fvp(const PdxPpoBatch* batch, const PdxMlp* pi, const float* log_std, const PdxMlp* dir,
                              float scale, float damping, const PdxMlpGrad* out, void* scratch, int64_t scratch_bytes,
                              void* stream) {
  using namespace pdx;
  if (!batch_ok(batch))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: batch needs n >= 1, 1 <= obs_dim <= 384 and obs");
  if (!mlp_ok(pi, 4) || !log_std)
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: actor must have two hidden layers of <= 64 units, 4 outputs and log_std");
  if (!mlp_ok(dir, 4) || dir->hidden[0] != pi->hidden[0] || dir->hidden[1] != pi->hidden[1])
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: dir must have the actor's shape and all six tensors");
  if (!out || !grad_ok(out))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: out needs all six tensors");
  // out must not overlap dir: k_ppo_fvp_reduce reads dir while it writes out
  const int64_t D = batch->obs_dim, h1 = pi->hidden[0], h2 = pi->hidden[1];
  const int64_t rows[3] = {h1, h2, 4}, cols[3] = {D, h1, h2};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) {
      const uintptr_t o = (uintptr_t)(i < 3 ? (const void*)out->weight[i] : (const void*)out->bias[i - 3]);
      const uintptr_t d = (uintptr_t)(j < 3 ? (const void*)dir->weight[j] : (const void*)dir->bias[j - 3]);
      const uintptr_t no = 4 * (uintptr_t)(i < 3 ? rows[i] * cols[i] : rows[i - 3]);
      const uintptr_t nd = 4 * (uintptr_t)(j < 3 ? rows[j] * cols[j] : rows[j - 3]);
      if (o < d + nd && d < o + no) return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: out must not alias dir");
    }
  if (!std::isfinite(scale) || !(damping >= 0.0f) || !std::isfinite(damping))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_pi_fvp: scale must be finite, damping finite and >= 0");
  return ppo_run("pdx_ppo_pi_fvp", kFvp, batch, pi, log_std, 0.0f, out, nullptr, nullptr, nullptr, nullptr, dir, scale,
                 damping, scratch, scratch_bytes, stream);
}

extern "C" int pdx_ppo_v_grad(const PdxPpoBatch* batch, const PdxMlp* v, const PdxMlpGrad* grad, float* loss,
                              void* scratch, int64_t scratch_bytes, void* stream) {
  using namespace pdx;
  if (!batch_ok(batch) || !batch->target_v)
    return set_error(PDX_ERR_INVALID, "pdx_ppo_v_grad: batch needs n >= 1, 1 <= obs_dim <= 384, obs and target_v");
  if (!mlp_ok(v, 1))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_v_grad: critic must have two hidden layers of <= 64 units and one output");
  if (!loss || !grad || !grad_ok(grad))
    return set_error(PDX_ERR_INVALID, "pdx_ppo_v_grad: loss and a gradient with all six tensors are required");
  return ppo_run("pdx_ppo_v_grad", kCritic, batch, v, nullptr, 0.0f, grad, loss, nullptr, nullptr, nullptr, nullptr, 0.0f, 0.0f,
                 scratch, scratch_bytes, stream);
}
