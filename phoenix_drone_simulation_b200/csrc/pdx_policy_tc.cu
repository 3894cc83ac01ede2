// ActorCritic.step (algs/core.py:370-393) on the 5th-generation tensor cores: tcgen05.mma with the
// accumulators -- and the hidden activations -- resident in tensor memory (TMEM).
//
//   standardise (utils/online_mean_std.py:42-48) -> actor MLP (relu, core.py:227-289) and critic MLP
//   (tanh, core.py:297-310) -> a = mu + exp(log_std) * N(0,1) (Philox) -> log-probability
//
// One CTA works on tiles of 128 environments: environment m of the tile is TMEM lane m and row m
// of every MMA (M = 128), so "one thread = one environment" holds for all element-wise work.
//
//   stage     raw observation tile (128 x D floats, contiguous in global memory) -> shared memory by
//             ONE bulk copy of the TMA engine; threads standardise it into the canonical K-major
//             operand layout X (tf32 hi / lo)
//   layer 1   D1[128 x 128] = 1 * b1 + X[128 x K1] * B1   SS: X and B1 in shared memory; columns 0..63
//                                                          actor, 64..127 critic.  The bias enters as
//                                                          the first MMA of the chain: a constant
//                                                          "ones" operand times a bias tile
//   epilogue  a2 = act(D1)  written back IN PLACE into the TMEM columns of D1
//   layer 2   D2[:, 0:64] = 1 * b2a + a2[:, 0:64] * B2a ; D2[:, 64:128] = 1 * b2c + a2[:, 64:128] * B2c
//                                                          TS: A operand read from TMEM.  Independent
//                                                          accumulators (actor / critic, and for the
//                                                          split mode two K halves each) are issued
//                                                          interleaved: a chain of MMAs into ONE
//                                                          accumulator runs at the MMA latency
//   epilogue  a3 = act(D2) stays in registers; layer 3 (64 x 4 + 64 x 1 weights) is a dot product on
//             the CUDA cores in float32 -- each thread covers its columns, partial sums meet in
//             shared memory -- then Philox draw, action, log-probability, stores
//
// The hidden activations never touch shared or global memory.  Every warp owns 32 TMEM lanes
// (lane quarter w & 3) and an equal share of actor (relu) and critic (tanh) columns.  Thread 0
// issues every tcgen05.mma and commits each layer to its own mbarrier.
//
// Precision: kind::tf32 keeps 10 explicit mantissa bits of each operand.  precision = 1 rounds the
// operands once (to nearest) -> ~1e-3 relative error on mu / v.  precision = 3 splits both operands
// x = hi + lo (hi = tf32(x), lo = x - hi) and accumulates A_lo*B_hi + A_hi*B_lo + A_hi*B_hi into the
// same fp32 TMEM accumulator (the dropped lo*lo term is 2^-22 relative): float32-level results at
// three times the (cheap) MMA cost, which is what the parity tests pin against torch.
#include "pdx_host.h"
#include "pdx_math.cuh"
#include "pdx_tc.cuh"

namespace {

struct TcArgs {
  int64_t n;
  int32_t obs_dim, k1, act_dim, flags;
  const float* obs;
  const float* mean;
  const float* std;
  float eps;
  const float* log_std;
  const float* packed;
  uint64_t seed, counter;
  int64_t env_offset;
  float* act; float* val; float* logp; float* mu;
  int64_t n_tiles;
};

// ---------------------------------------------------------------------------------------------
//  Packed weight image (global == shared layout), floats:
//    common  w3a[64][4] (actor output weights, [hidden][action]), w3c[64] (critic), b3[16] (mu biases 0..3, v bias 4)
//    Bhi     B1[K1/4][128][4]  B2a[16][64][4]  B2c[16][64][4]  Bc[2][64][4] (pdx_collect's critic layer-2 bias tile)
//            bias tiles  Bb1[2][128][4]  Bb2a[2][64][4]  Bb2c[2][64][4]                  (tf32-rounded)
//    Blo     same shapes, w - hi                                                  (precision 3 only)
//  B?[kc][n][j] = W[n][4 kc + j]  (torch nn.Linear weight is [out][in]): exactly the no-swizzle K-major
//  core-matrix layout with SBO = 128 B and LBO = 16 N bytes.  Bb?[0][n][0] = bias[n], rest zero.
// ---------------------------------------------------------------------------------------------

struct PackArgs {
  int32_t obs_dim, k1, x3;
  int32_t pi_h1, pi_h2, v_h1, v_h2, act_dim;
  const float* pi_w[3]; const float* pi_b[3];
  const float* v_w[3]; const float* v_b[3];
  float* out;
};

__global__ void k_pack_tc(const PackArgs a) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  const int D = a.obs_dim, K1 = a.k1;
  float* common = a.out;
  float* bhi = common + kCommonWords;
  float* blo = bhi + tc_b_words(K1);
  for (int j = tid; j < kCommonWords; j += nt) {
    float w = 0.0f;
    if (j < 256) { const int k = j >> 2, o = j & 3; if (k < a.pi_h2 && o < a.act_dim) w = a.pi_w[2][o * a.pi_h2 + k]; }
    else if (j < 320) { if (j - 256 < a.v_h2) w = a.v_w[2][j - 256]; }
    else if (j - 320 < a.act_dim) w = a.pi_b[2][j - 320];
    else if (j - 320 == 4) w = a.v_b[2][0];
    common[j] = w;
  }
  const int total = (int)tc_b_words(K1);
  for (int idx = tid; idx < total; idx += nt) {
    float w = 0.0f;
    int r = idx;
    if (r < K1 * kN1) {                                   // B1: N = 128
      const int kc = r / (kN1 * 4), n = (r / 4) % kN1, k = 4 * kc + (r & 3);
      if (k < D) {
        if (n < 64) { if (n < a.pi_h1) w = a.pi_w[0][n * D + k]; }
        else if (n - 64 < a.v_h1) w = a.v_w[0][(n - 64) * D + k];
      } else if (k == D) {                                // the constant-1 column of X (pdx_collect): layer-1 biases, and
        if (n < 64) {                                     // a constant-1 hidden unit after the actor's last one
          if (n < a.pi_h1) w = a.pi_b[0][n];
          else if (n == a.pi_h1) w = 1.0f;
        } else if (n - 64 < a.v_h1) w = a.v_b[0][n - 64];
      }
    } else if ((r -= K1 * kN1) < 2 * kB2Words) {          // B2a, B2c: N = 64, K = 64
      const bool critic = r >= kB2Words;
      if (critic) r -= kB2Words;
      const int kc = r / 256, n = (r / 4) % 64, k = 4 * kc + (r & 3);
      const int h1 = critic ? a.v_h1 : a.pi_h1, h2 = critic ? a.v_h2 : a.pi_h2;
      if (n < h2 && k < h1) w = (critic ? a.v_w[1] : a.pi_w[1])[n * h1 + k];
      else if (!critic && n < h2 && k == h1) w = a.pi_b[1][n];      // (h1 < 64) the constant-1 unit's row: actor layer-2 bias
    } else if ((r -= 2 * kB2Words) < kColBiasWords) {     // pdx_collect: extra K step of the critic's layer 2 over the
      const int kc = r / 256, n = (r / 4) % 64, k = 4 * kc + (r & 3);   // actor columns 8 (pi_h1 / 8) ..: constant-1 unit
      if (a.pi_h1 < 64 && k == (a.pi_h1 & 7) && n < a.v_h2) w = a.v_b[1][n];
    } else {                                              // bias tiles: only element (kc = 0, n, j = 0) is non-zero
      r -= kColBiasWords;
      if (r < 8 * kN1) {
        const int n = r / 4;
        if ((r & 3) == 0 && n < kN1) { if (n < 64) { if (n < a.pi_h1) w = a.pi_b[0][n]; } else if (n - 64 < a.v_h1) w = a.v_b[0][n - 64]; }
      } else if ((r -= 8 * kN1) < 8 * 64) {
        const int n = r / 4;
        if ((r & 3) == 0 && n < 64 && n < a.pi_h2) w = a.pi_b[1][n];
      } else {
        r -= 8 * 64;
        const int n = r / 4;
        if ((r & 3) == 0 && n < 64 && n < a.v_h2) w = a.v_b[1][n];
      }
    }
    const float hi = __uint_as_float(tf32_rna(w));
    bhi[idx] = hi;
    if (a.x3) blo[idx] = w - hi;
  }
}

// ---------------------------------------------------------------------------------------------
//  The kernel
// ---------------------------------------------------------------------------------------------
#ifdef PDX_TC_TIMING
__device__ long long tc_timing[16 * 8];
#define TC_STAMP(slot) do { if (blockIdx.x == 0 && tid == 64 && tcount < 8) tc_timing[tcount * 16 + (slot)] = clock64(); } while (0)
#else
#define TC_STAMP(slot) do { } while (0)
#endif

template <bool X3>
struct TcCfg {
  static constexpr int kThreads = X3 ? 512 : 256;      // X3: one CTA per SM (TMEM), 16 warps; else two CTAs of 8 warps
  static constexpr int kNcg = kThreads / 128;          // column groups: warps w, w+4, ... share TMEM lane quarter w & 3
  static constexpr int kCw = 64 / kNcg;                // columns per net and thread (16 or 32)
  static constexpr int kTmemCols = X3 ? 512 : 256;
  static constexpr int kMinBlocks = X3 ? 1 : 2;
  static constexpr int kSplit = 1;                     // layer-2 accumulators per net (2 = K halves summed in the epilogue: no gain measured)
  // TMEM column regions: R0 = D1 -> a2 (hi), R1 = D2 (first K half), R2 = a2 lo, R3 = D2 (second K half)
  static constexpr uint32_t kR0 = 0, kR1 = 128, kR2 = 256, kR3 = 384;     // kR3 only with kSplit = 2
};

// a2 = act(D1) for this thread's 2 x CW columns, written back in place as layer 2's A operand (hi) and,
// for X3, the lo halves into region R2.
template <bool X3>
__device__ __forceinline__ void hidden_epilogue(uint32_t taddr, int cg) {
  using Cfg = TcCfg<X3>;
#pragma unroll
  for (int c = 0; c < Cfg::kCw / 16; ++c) {
    const int ca = cg * Cfg::kCw + 16 * c, cc = 64 + ca;            // actor / critic column of this chunk
    uint32_t ra[16], rc[16], la[16], lc[16];
    tmem_ld16(taddr + Cfg::kR0 + ca, ra);
    tmem_ld16(taddr + Cfg::kR0 + cc, rc);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float ya = fmaxf(__uint_as_float(ra[j]), 0.0f);
      const float xc = __uint_as_float(rc[j]);
      const float yc = X3 ? tanh_fast(xc) : tanh_mufu(xc);
      ra[j] = tf32_rna(ya);
      rc[j] = tf32_rna(yc);
      if (X3) {
        la[j] = __float_as_uint(ya - __uint_as_float(ra[j]));
        lc[j] = __float_as_uint(yc - __uint_as_float(rc[j]));
      }
    }
    tmem_st16(taddr + Cfg::kR0 + ca, ra);
    tmem_st16(taddr + Cfg::kR0 + cc, rc);
    if (X3) {
      tmem_st16(taddr + Cfg::kR2 + ca, la);
      tmem_st16(taddr + Cfg::kR2 + cc, lc);
    }
  }
}

// a3 = act(D2) for this thread's columns and its share of layer 3 in float32:
// part[0..3] += a3_actor[col] * w3a[col][0..3], part[4] += a3_critic[col] * w3c[col]
template <bool X3>
__device__ __forceinline__ void output_epilogue(uint32_t taddr, int cg, const float* __restrict__ w3a,
                                                const float* __restrict__ w3c, float (&part)[5]) {
  using Cfg = TcCfg<X3>;
#pragma unroll
  for (int k = 0; k < 5; ++k) part[k] = 0.0f;
#pragma unroll
  for (int c = 0; c < Cfg::kCw / 16; ++c) {
    const int ca = cg * Cfg::kCw + 16 * c, cc = 64 + ca;
    uint32_t ra[16], rc[16];
    tmem_ld16(taddr + Cfg::kR1 + ca, ra);
    tmem_ld16(taddr + Cfg::kR1 + cc, rc);
    if (Cfg::kSplit == 2) {
      uint32_t sa[16], sc[16];
      tmem_ld16(taddr + Cfg::kR3 + ca, sa);
      tmem_ld16(taddr + Cfg::kR3 + cc, sc);
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        ra[j] = __float_as_uint(__uint_as_float(ra[j]) + __uint_as_float(sa[j]));
        rc[j] = __float_as_uint(__uint_as_float(rc[j]) + __uint_as_float(sc[j]));
      }
    } else {
      tmem_wait_ld();
    }
    float wc[16];
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {                       // ca is a multiple of 16: 128-bit broadcast loads
      const float4 t = *reinterpret_cast<const float4*>(w3c + ca + 4 * j4);
      wc[4 * j4] = t.x; wc[4 * j4 + 1] = t.y; wc[4 * j4 + 2] = t.z; wc[4 * j4 + 3] = t.w;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float ya = fmaxf(__uint_as_float(ra[j]), 0.0f);
      const float xc = __uint_as_float(rc[j]);
      const float yc = X3 ? tanh_fast(xc) : tanh_mufu(xc);
      const float4 w = *reinterpret_cast<const float4*>(w3a + 4 * (ca + j));
      part[0] = fmaf(ya, w.x, part[0]);
      part[1] = fmaf(ya, w.y, part[1]);
      part[2] = fmaf(ya, w.z, part[2]);
      part[3] = fmaf(ya, w.w, part[3]);
      part[4] = fmaf(yc, wc[j], part[4]);
    }
  }
}

template <bool X3>
__global__ void __launch_bounds__(TcCfg<X3>::kThreads + 32, TcCfg<X3>::kMinBlocks) k_policy_tc(const TcArgs a) {
  using Cfg = TcCfg<X3>;
  constexpr int NT = Cfg::kThreads;                                        // epilogue threads; warp NT/32 is the issuer
  constexpr int NB = X3 ? 2 : 1;                                           // operand images: hi (+ lo)
  constexpr uint32_t R0 = Cfg::kR0, R1 = Cfg::kR1, R2 = Cfg::kR2;
  constexpr int kBarEpi = 1, kBarA2 = 2, kBarX = 3;                        // named barriers (0 = __syncthreads)
  extern __shared__ __align__(128) uint8_t tc_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = a.obs_dim, K1 = a.k1;
  const bool issuer = warp == NT / 32;

  // ---- shared-memory plan
  uint64_t* mbar = reinterpret_cast<uint64_t*>(tc_smem);                   // [0] weights [1..2] layers [3] obs tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tc_smem + 40);
  float* act_std = reinterpret_cast<float*>(tc_smem + 48);                 // exp(log_std)[4], then log_std[4]
  float2* norm = reinterpret_cast<float2*>(tc_smem + 80);                  // [K1] (mean, 1/(std+eps))
  uint8_t* ones = tc_smem + 80 + K1 * 8;                                   // constant A operand: column 0 = 1
  float* part_sm = reinterpret_cast<float*>(ones + kOnesBytes);            // [kNcg][128][8] layer-3 partial sums
  float* common = part_sm + Cfg::kNcg * kTile * 8;                         // w3a, w3c, b3 (start of the weight image)
  float* bhi = common + kCommonWords;
  const int64_t bwords = tc_b_words(K1);
  uint8_t* a1hi = reinterpret_cast<uint8_t*>(bhi + NB * bwords);
  uint8_t* a1lo = a1hi + (K1 / 4) * kLboA;
  float* stage = reinterpret_cast<float*>(a1hi + NB * (K1 / 4) * kLboA);   // raw observation tile [128][D]
  const uint32_t bar_w = smem_u32(mbar), bar1 = bar_w + 8, bar2 = bar_w + 16, bar_x = bar_w + 24;

  if (!(a.flags & 1)) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }
  // ---- one-time setup (all warps)
  if (warp == 0) tmem_alloc<Cfg::kTmemCols>(smem_u32(tmem_slot));
  if (tid == 32) {
    mbar_init(bar_w, 1); mbar_init(bar1, 1); mbar_init(bar2, 1); mbar_init(bar_x, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 4) {
    const float ls = tid < a.act_dim ? a.log_std[tid] : 0.0f;
    act_std[tid] = expf(ls);
    act_std[4 + tid] = ls;
  }
  for (int k = tid; k < K1; k += NT + 32) {
    float m = 0.0f, inv = 1.0f;
    if (k < D && a.std) { m = a.mean[k]; inv = 1.0f / (a.std[k] + a.eps); }
    norm[k] = make_float2(m, inv);
  }
  for (int e = tid; e < (int)kOnesBytes / 4; e += NT + 32)                  // ones[m][k]: k = 0 -> 1
    reinterpret_cast<float*>(ones)[e] = (e < 512 && (e & 3) == 0) ? 1.0f : 0.0f;
  const int n_chunks = (D + 3) >> 2;                                        // 16-byte K chunks that hold data
  for (int e = tid; e < kTile * (K1 / 4 - n_chunks); e += NT + 32) {        // K padding chunks: zero, once
    const int m = e & (kTile - 1), kc = n_chunks + (e >> 7);
    *reinterpret_cast<float4*>(a1hi + kc * kLboA + m * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
    if (X3) *reinterpret_cast<float4*>(a1lo + kc * kLboA + m * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  fence_async_smem();                // ones / padding (generic proxy) -> visible to the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_slot;
  // Programmatic dependent launch: everything above may run while the kernel before this one on the stream
  // drains.  PDX_POLICY_TC_OVERLAP (flags bit 0) is the caller's promise that that kernel writes none of
  // log_std / normaliser / weight image, which were read above / are staged below; without the promise
  // the wait sits at the top of the kernel.  Observations are only fetched after the wait.
  if (a.flags & 1) {
    if (issuer && lane == 0) {         // weight image: one bulk copy, under the predecessor's tail
      const uint32_t bytes = (uint32_t)((kCommonWords + NB * bwords) * 4);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_w), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(common)),
                   "l"(a.packed), "r"(bytes), "r"(bar_w)
                   : "memory");
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }
  const bool obs_aligned = (reinterpret_cast<uintptr_t>(a.obs) & 15) == 0;
  // a tile travels by ONE bulk copy (TMA engine) when it is complete and 16-byte aligned; the last,
  // partial tile is copied by the epilogue threads themselves
  auto tile_is_bulk = [&](int64_t tile) { return (a.n - tile * kTile) >= kTile && obs_aligned; };

  if (issuer) {
    // =====================================================================================
    //  issuer warp: TMA copies and every tcgen05.mma.  All 32 lanes run this code with
    //  warp-uniform values; the wrappers elect the lane that executes the instruction.
    // =====================================================================================
    const uint32_t b1_s = smem_u32(bhi), b2a_s = b1_s + K1 * kN1 * 4, b2c_s = b2a_s + kB2Words * 4;
    const uint32_t bb1_s = b2c_s + (kB2Words + kColBiasWords) * 4, bb2a_s = bb1_s + 8 * kN1 * 4, bb2c_s = bb2a_s + 8 * 64 * 4;
    const uint32_t lo_off = (uint32_t)bwords * 4;          // Blo = Bhi + lo_off (bytes)
    const uint32_t a1hi_s = smem_u32(a1hi), a1lo_s = smem_u32(a1lo);
    const uint64_t ones_desc = make_desc(smem_u32(ones), 2048, kSbo);
    auto fetch = [&](int64_t tile) {
      if (tile < a.n_tiles && tile_is_bulk(tile) && lane == 0) {
        const uint32_t bytes = (uint32_t)(kTile * D * 4);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_x), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(stage)),
                     "l"(a.obs + tile * kTile * D), "r"(bytes), "r"(bar_x)
                     : "memory");
      }
      __syncwarp();
    };
    // descriptors advance by two K chunks per MMA (K = 8 tf32): the 14-bit address field never carries
    auto issue_layer1 = [&]() {
      constexpr uint32_t idesc = make_idesc(kN1);
      constexpr uint32_t lbo_b = kN1 * 16;
      mma_ss(tbase + R0, ones_desc, make_desc(bb1_s, lbo_b, kSbo), idesc, 0);
      if (X3) mma_ss(tbase + R0, ones_desc, make_desc(bb1_s + lo_off, lbo_b, kSbo), idesc, 1);
      uint64_t ah = make_desc(a1hi_s, kLboA, kSbo), al = make_desc(a1lo_s, kLboA, kSbo);
      uint64_t bh = make_desc(b1_s, lbo_b, kSbo), bl = make_desc(b1_s + lo_off, lbo_b, kSbo);
#pragma unroll 1
      for (int ks = 0; ks < K1 / 8; ++ks) {
        if (X3) {
          mma_ss(tbase + R0, al, bh, idesc, 1);
          mma_ss(tbase + R0, ah, bl, idesc, 1);
        }
        mma_ss(tbase + R0, ah, bh, idesc, 1);
        ah += (2 * kLboA) >> 4; al += (2 * kLboA) >> 4; bh += (2 * lbo_b) >> 4; bl += (2 * lbo_b) >> 4;
      }
      tc_commit(bar1);
    };
    auto issue_layer2 = [&]() {
      constexpr uint32_t idesc = make_idesc(64);
      constexpr uint32_t lbo_b = 64 * 16;
      constexpr uint64_t kstep = (2 * lbo_b) >> 4;
      uint64_t bha = make_desc(b2a_s, lbo_b, kSbo), bhc = make_desc(b2c_s, lbo_b, kSbo);
      uint64_t bla = make_desc(b2a_s + lo_off, lbo_b, kSbo), blc = make_desc(b2c_s + lo_off, lbo_b, kSbo);
      mma_ss(tbase + R1, ones_desc, make_desc(bb2a_s, lbo_b, kSbo), idesc, 0);
      mma_ss(tbase + R1 + 64, ones_desc, make_desc(bb2c_s, lbo_b, kSbo), idesc, 0);
      if (X3) {
        mma_ss(tbase + R1, ones_desc, make_desc(bb2a_s + lo_off, lbo_b, kSbo), idesc, 1);
        mma_ss(tbase + R1 + 64, ones_desc, make_desc(bb2c_s + lo_off, lbo_b, kSbo), idesc, 1);
      }
      // rolled over the k-steps; within a step the two nets' (independent) accumulators alternate
      uint32_t a_hi = tbase + R0, a_lo = tbase + R2;
#pragma unroll 1
      for (int ks = 0; ks < 8; ++ks) {
        if (X3) {
          mma_ts(tbase + R1, a_lo, bha, idesc, 1);
          mma_ts(tbase + R1 + 64, a_lo + 64, bhc, idesc, 1);
          mma_ts(tbase + R1, a_hi, bla, idesc, 1);
          mma_ts(tbase + R1 + 64, a_hi + 64, blc, idesc, 1);
        }
        mma_ts(tbase + R1, a_hi, bha, idesc, 1);
        mma_ts(tbase + R1 + 64, a_hi + 64, bhc, idesc, 1);
        a_hi += 8; a_lo += 8; bha += kstep; bhc += kstep; bla += kstep; blc += kstep;
      }
      tc_commit(bar2);
    };

    int64_t tile = blockIdx.x;
    if (lane == 0 && !(a.flags & 1)) {                     // weight image: one bulk copy
      const uint32_t bytes = (uint32_t)((kCommonWords + NB * bwords) * 4);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_w), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(common)),
                   "l"(a.packed), "r"(bytes), "r"(bar_w)
                   : "memory");
    }
    __syncwarp();
    fetch(tile);
    named_bar_sync(kBarX, NT + 32);                        // X(tile 0) built, `stage` consumed
    fetch(tile + gridDim.x);
    mbar_wait(bar_w, 0);
    tc_fence_after();
    issue_layer1();
    uint32_t par = 0;
    for (; tile < a.n_tiles; tile += gridDim.x, par ^= 1) {
      const int64_t next = tile + gridDim.x;
      named_bar_sync(kBarA2, NT + 32);                     // a2 of this tile is in TMEM
      tc_fence_after();
      issue_layer2();
      if (next < a.n_tiles) {
        named_bar_sync(kBarX, NT + 32);                    // X(next) built, `stage` consumed
        fetch(next + gridDim.x);
        mbar_wait(bar2, par);                              // layer 2 has read a2: its columns are free for D1(next)
        tc_fence_after();
        issue_layer1();
      }
    }
  } else {
    // =====================================================================================
    //  epilogue warps: element-wise work, one thread = one environment row of the tile
    // =====================================================================================
    const int q = warp & 3, cg = warp >> 2;                // TMEM lane quarter, column group
    const uint32_t taddr = tbase + ((uint32_t)(32 * q) << 16);
    const int row = 32 * q + lane;                         // this thread's environment within the tile
    const float* w3a = common;
    const float* w3c = common + 256;
    const float* b3 = common + 320;
    // raw tile in `stage` (bulk copy signalled on bar_x, or copied here) -> X: standardise, split, store in
    // the canonical K-major layout.  Sixteen lanes walk the 16-byte K chunks of one environment row
    // (contiguous shared-memory reads), two rows per warp.
    auto build_x = [&](int64_t tile, uint32_t parity) {
      if (tile_is_bulk(tile)) {
        mbar_wait(bar_x, parity);
      } else {
        const int64_t env0 = tile * kTile;
        const int n_elem = (int)(((a.n - env0) < kTile ? (a.n - env0) : kTile) * D);
        const float* src = a.obs + env0 * D;
        for (int e = tid; e < kTile * D; e += NT) stage[e] = e < n_elem ? __ldg(src + e) : 0.0f;
        named_bar_sync(kBarEpi, NT);
      }
      const int kc = tid & 15;
      if (kc < n_chunks) {
        float2 nm[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) nm[j] = 4 * kc + j < D ? norm[4 * kc + j] : make_float2(0.0f, 0.0f);
#pragma unroll 4
        for (int m = tid >> 4; m < kTile; m += NT / 16) {
          const float* src = stage + m * D + 4 * kc;
          uint32_t hi[4];
          float lo[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float x = 4 * kc + j < D ? (src[j] - nm[j].x) * nm[j].y : 0.0f;
            hi[j] = tf32_rna(x);
            lo[j] = x - __uint_as_float(hi[j]);
          }
          *reinterpret_cast<uint4*>(a1hi + kc * kLboA + m * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          if (X3) *reinterpret_cast<float4*>(a1lo + kc * kLboA + m * 16) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_async_smem();            // generic-proxy writes of X -> visible to the tensor core (async proxy)
      named_bar_arrive(kBarX, NT + 32);
    };

    int64_t tile = blockIdx.x;
    build_x(tile, 0);
    mbar_wait(bar_w, 0);             // layer-3 weights / biases are read from the image below
    uint32_t par = 0;
    [[maybe_unused]] int tcount = 0;
    for (; tile < a.n_tiles; tile += gridDim.x, par ^= 1, ++tcount) {
      const int64_t env0 = tile * kTile;
      const int64_t next = tile + gridDim.x;
      // ---- layer 1 done -> activation in place (TMEM), hand a2 to the issuer
      TC_STAMP(0);
      mbar_wait(bar1, par);
      tc_fence_after();
      TC_STAMP(1);
      hidden_epilogue<X3>(taddr, cg);
      tmem_wait_st();
      tc_fence_before();
      named_bar_arrive(kBarA2, NT + 32);
      TC_STAMP(2);
      // ---- while layer 2 runs: the next tile's observations -> X (layer 1 of this tile has completed,
      // so the X buffer is free)
      if (next < a.n_tiles) build_x(next, par ^ 1);
      TC_STAMP(3);
      // the Gaussian draw does not depend on the networks: do it now, while layer 2 runs, instead of on the
      // critical path after the last epilogue.  Same Philox counters as k_policy: identical draws for the
      // same (seed, counter, env).
      float eps[4] = {0.f, 0.f, 0.f, 0.f}, lp = 0.0f;
      if (cg == 0) {
        pdx::policy_normals(a.seed, a.counter, (uint64_t)(a.env_offset + env0 + row), eps);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (k < a.act_dim) lp += -0.5f * eps[k] * eps[k] - act_std[4 + k] - 0.9189385332046727f;
      }
      // ---- layer 2 done -> activation, layer 3 partial dot products
      mbar_wait(bar2, par);
      tc_fence_after();
      TC_STAMP(4);
      float part[5];
      output_epilogue<X3>(taddr, cg, w3a, w3c, part);
      {
        float4* dst = reinterpret_cast<float4*>(part_sm + (cg * kTile + row) * 8);
        dst[0] = make_float4(part[0], part[1], part[2], part[3]);
        dst[1] = make_float4(part[4], 0.f, 0.f, 0.f);
      }
      tc_fence_before();
      TC_STAMP(5);
      named_bar_sync(kBarEpi, NT);
      TC_STAMP(6);
      // ---- output: mu, v = bias + partial sums; sample, log-probability, stores
      if (cg == 0) {
        const int64_t i = env0 + row;
        if (i < a.n) {
          float mu[4] = {b3[0], b3[1], b3[2], b3[3]};
          float v = b3[4];
#pragma unroll
          for (int g = 0; g < Cfg::kNcg; ++g) {
            const float4* src = reinterpret_cast<const float4*>(part_sm + (g * kTile + row) * 8);
            const float4 p0 = src[0];
            mu[0] += p0.x; mu[1] += p0.y; mu[2] += p0.z; mu[3] += p0.w;
            v += src[1].x;
          }
          float av[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < a.act_dim) av[k] = fmaf(act_std[k], eps[k], mu[k]);
          reinterpret_cast<float4*>(a.act)[i] = make_float4(av[0], av[1], av[2], av[3]);
          a.val[i] = v;
          a.logp[i] = lp;
          if (a.mu) reinterpret_cast<float4*>(a.mu)[i] = make_float4(mu[0], mu[1], mu[2], mu[3]);
        }
      }
      TC_STAMP(7);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_free<Cfg::kTmemCols>(tbase);
}

size_t tc_smem_bytes(int k1, int obs_dim, bool x3) {
  const size_t nb = x3 ? 2 : 1, ncg = x3 ? 4 : 2;
  return 80 + (size_t)k1 * 8 + kOnesBytes + ncg * kTile * 8 * 4 + (kCommonWords + nb * tc_b_words(k1)) * 4 +
         nb * (k1 / 4) * kLboA + (size_t)kTile * obs_dim * 4;
}

bool tc_shapes_ok(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, int32_t precision) {
  if (obs_dim <= 0 || !pi || !v || (precision != 1 && precision != 3)) return false;
  if (pi->hidden[0] < 1 || pi->hidden[0] > 64 || pi->hidden[1] < 1 || pi->hidden[1] > 64 || pi->n_out < 1 || pi->n_out > 4) return false;
  if (v->hidden[0] < 1 || v->hidden[0] > 64 || v->hidden[1] < 1 || v->hidden[1] > 64 || v->n_out != 1) return false;
  const int k1 = tc_k1(obs_dim);
  if (k1 > 64) return false;                              // sixteen lanes walk the K chunks of a row (stage_to_x)
  return tc_smem_bytes(k1, obs_dim, precision == 3) <= pdx::kMaxSmemBytes;
}

}  // namespace

#ifdef PDX_TC_TIMING
extern "C" int pdx_policy_tc_timing(long long* out) {
  return cudaMemcpyFromSymbol(out, tc_timing, sizeof(long long) * 128) == cudaSuccess ? 0 : -2;
}
#endif

extern "C" int64_t pdx_policy_tc_pack_words(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, int32_t precision) {
  if (!tc_shapes_ok(obs_dim, pi, v, precision))
    return pdx::set_error(PDX_ERR_INVALID, "tensor-core policy plan: needs two hidden layers <= 64, n_out <= 4, obs_dim <= 64, precision 1 or 3");
  const int k1 = tc_k1(obs_dim);
  return kCommonWords + (precision == 3 ? 2 : 1) * tc_b_words(k1);
}

extern "C" int pdx_policy_tc_pack(int32_t obs_dim, const PdxMlp* pi, const PdxMlp* v, int32_t precision, float* packed, void* stream) {
  if (!packed || !tc_shapes_ok(obs_dim, pi, v, precision))
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_tc_pack: null buffer or shapes outside the tensor-core plan");
  const int rc = pdx::select_device_of(packed);
  if (rc) return rc;
  PackArgs p;
  p.obs_dim = obs_dim; p.k1 = tc_k1(obs_dim); p.x3 = precision == 3;
  p.pi_h1 = pi->hidden[0]; p.pi_h2 = pi->hidden[1]; p.v_h1 = v->hidden[0]; p.v_h2 = v->hidden[1]; p.act_dim = pi->n_out;
  for (int k = 0; k < 3; ++k) { p.pi_w[k] = pi->weight[k]; p.pi_b[k] = pi->bias[k]; p.v_w[k] = v->weight[k]; p.v_b[k] = v->bias[k]; }
  p.out = packed;
  k_pack_tc<<<16, 256, 0, (cudaStream_t)stream>>>(p);
  return pdx::cuda_error("pdx_policy_tc_pack", cudaGetLastError());
}

extern "C" int pdx_policy_step_tc(int64_t n, int32_t obs_dim, const float* obs, const float* mean, const float* std, float eps,
                                  const PdxMlp* pi, const PdxMlp* v, const float* log_std, const float* packed, int32_t precision,
                                  uint64_t seed, uint64_t counter, int64_t env_offset, float* actions, float* values, float* logp,
                                  float* mu_out, void* stream) {
  const int32_t overlap = (precision & PDX_POLICY_TC_OVERLAP) ? 1 : 0;
  precision &= ~PDX_POLICY_TC_OVERLAP;
  if (n <= 0 || !obs || !log_std || !packed || !actions || !values || !logp || !tc_shapes_ok(obs_dim, pi, v, precision))
    return pdx::set_error(PDX_ERR_INVALID, "pdx_policy_step_tc: null buffer, n <= 0 or shapes outside the tensor-core plan");
  int dev = 0;
  int rc = pdx::select_device_of(obs, &dev);
  if (rc) return rc;
  const bool x3 = precision == 3;
  TcArgs a;
  a.n = n; a.obs_dim = obs_dim; a.k1 = tc_k1(obs_dim); a.act_dim = pi->n_out;
  a.flags = overlap;
  a.obs = obs; a.mean = mean; a.std = std; a.eps = eps; a.log_std = log_std; a.packed = packed;
  a.seed = seed; a.counter = counter; a.env_offset = env_offset; a.act = actions; a.val = values; a.logp = logp; a.mu = mu_out;
  a.n_tiles = (n + kTile - 1) / kTile;
  const size_t smem = tc_smem_bytes(a.k1, obs_dim, x3);
  auto kern = x3 ? k_policy_tc<true> : k_policy_tc<false>;
  rc = pdx::cuda_error("pdx_policy_step_tc (shared-memory opt-in)", pdx::opt_in_smem(kern, dev, smem));
  if (rc) return rc;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // persistent CTAs: TMEM (512 columns per SM) admits one precision-3 CTA or two precision-1 CTAs per SM
  const int64_t resident = (int64_t)sms * (x3 ? 1 : (2 * smem <= pdx::kMaxSmemBytes ? 2 : 1));
  const unsigned grid = (unsigned)(a.n_tiles < resident ? a.n_tiles : resident);
  // the grid may start while its predecessor drains (see the kernel)
  const int block = (x3 ? TcCfg<true>::kThreads : TcCfg<false>::kThreads) + 32;
  const cudaError_t e = pdx::launch_early(kern, grid, block, smem, (cudaStream_t)stream, true, a);
  return pdx::cuda_error("pdx_policy_step_tc", e != cudaSuccess ? e : cudaGetLastError());
}
