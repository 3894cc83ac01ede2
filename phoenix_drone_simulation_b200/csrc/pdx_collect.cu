// pdx_collect: the closed loop of IWPGAlgorithm.roll_out (algs/iwpg/iwpg.py:350-385) for a shard of
// lock-step environments in ONE persistent kernel:
//
//     for t in 0..T-1:   a, v, logp = ActorCritic.step(obs)      (algs/core.py:370-393)
//                        obs, r, terminated, truncated = env.step(a)   (envs/base.py:433-475, auto-reset)
//     last_val = V(obs)                                           (iwpg.py:376-378: the cut is bootstrapped)
//
// Design
//   * one CTA per SM; a CTA owns up to 14 warps x 32 environments for a whole pass of T steps, the
//     environment state stays in registers (rollout_step of pdx_kernels.cuh -- the same step body as
//     the open-loop kernel), its observation row in a per-warp shared-memory tile that leaves by bulk
//     copy.  Shards larger than one pass (148 CTAs x 448 envs) run further passes: environments are
//     independent, so "all steps of half the shard, then all steps of the other half" collects the same
//     rollout as lock-step order.
//   * a TILE = 4 warps = 128 environments = the 128 lanes of tensor memory = M of the MMAs.  The policy
//     step of a tile is tcgen05 work on a SLOT (a range of TMEM columns plus one operand buffer):
//     every thread standardises its own observation row into the K-major operand tile X, the tile's
//     first warp issues layer 1 (X . B1, both nets, N = 128), every thread runs the layer-1 epilogue of
//     ITS row (relu / tanh, TF32 rounding, written back to TMEM in place; the biases came in through a
//     constant-1 column of X, see tc_k1), layer 2 takes its A operand
//     from TMEM, and the layer-2 epilogue ends in the 64 x 4 + 64 dot products of layer 3, the Gaussian
//     draw and the log-probability -- the action never leaves the thread's registers on its way into
//     env.step.  There are no dedicated epilogue or issuer warps: while one tile waits for the tensor
//     pipe, the other tiles of the CTA are somewhere in their env.step.
//   * single-TF32 operands (precision 1): two slots of 256 columns; split-TF32 (precision 3, float32-level
//     results): one slot of 384 columns, the tiles of a CTA take turns.
//   * reset packages (pdx_kernels.cuh) are regenerated per tile (named-barrier vote of its 128 threads).
//
// Global traffic per env-step is the rollout itself: observation row, action, value, log-probability,
// reward, cost and the two flags.
#include "pdx_dispatch.cuh"
#include "pdx_tc.cuh"

// Measured slower on configs[4] (DESIGN.md §4): keeping two 16-column tcgen05.ld chunks in flight in the epilogues
// (software prefetch of the next chunk, 1,508 vs 1,420 us) -- more live registers and code for a latency the other
// tiles already cover.  Separate locks for the operand buffer X and the TMEM slot with one X buffer per tile (X built
// while other tiles hold the slots, buffer released after layer 1, per-tile mbarriers): 1,470 vs 1,400 us single
// TF32, 2,625 vs 2,295 us split TF32 -- every tile then queues for a slot at the same moment, where the single lock
// staggers the tiles by itself.  Skipping the actor's zero-weight hidden units in the layer-3 dot products behind
// uniform branches (+1.2 %).  No gain: the layer-3 dot products as packed FFMA2 (fma.rn.f32x2 with a broadcast
// scalar: half the FMA instructions, same time).

namespace pdx {

constexpr unsigned kSlotSpinNs = 40;         // back-off of the slot spin in ns (200: +1 % kernel time)

struct CollectArgs {
  int32_t obs_dim, k1, act_dim, n_steps;
  int32_t warps_per_cta, groups;             // environments per CTA and pass = 32 * warps_per_cta; groups of that size in the shard
  const float* obs0;                         // [n][D] observation the rollout starts from
  const float* mean; const float* std; float eps;
  const float* log_std;
  const float* packed;                       // weight image of pdx_policy_tc_pack (same precision)
  int32_t pi_h[2], v_h[2];
  uint64_t pol_seed, pol_counter;
  float* act; float* val; float* logp;       // [T][n][4], [T][n], [T][n]
  float* last_val;                           // [n]
  unsigned char* scratch;                    // per-thread episode-statistics columns of every CTA (global memory)
  double* obs_moments;                       // optional [2][D]: sum (o - mean), sum (o - mean)^2 over the T x n policy inputs
};

template <bool X3>
struct ColCfg {
  static constexpr int kSlots = X3 ? 1 : 2;
  static constexpr int kSlotCols = X3 ? 384 : 256;
  static constexpr int kImages = X3 ? 2 : 1;           // operand images: hi (+ lo)
  static constexpr uint32_t kR0 = 0, kR1 = 128, kR2 = 256;
};

__host__ __device__ inline int64_t collect_w_words(int k1) { return (int64_t)k1 * kN1 + 2 * kB2Words + kColBiasWords; }   // B1, B2a, B2c, Bc of one image

// shared-memory plan (bytes), in this order
struct ColSmem {
  size_t ctrl, norm, common, weights, x, tiles, moments, total;
};
template <bool X3>
__host__ __device__ inline ColSmem collect_smem(int k1, int D, int warps) {
  ColSmem s;
  s.ctrl = 0;                                          // 256 bytes of barriers / slot bookkeeping
  s.norm = 256;
  s.common = s.norm + (size_t)k1 * 8;
  s.common = (s.common + 15) & ~(size_t)15;
  s.weights = s.common + (size_t)kCommonWords * 4;
  s.x = s.weights + (size_t)ColCfg<X3>::kImages * collect_w_words(k1) * 4;
  s.x = (s.x + 127) & ~(size_t)127;
  s.tiles = s.x + (size_t)ColCfg<X3>::kSlots * ColCfg<X3>::kImages * (k1 / 4) * kLboA;
  s.tiles = (s.tiles + 15) & ~(size_t)15;
  s.moments = (s.tiles + (size_t)warps * 32 * D * 4 + 15) & ~(size_t)15;
  s.total = s.moments + (size_t)warps * 2 * 64 * 8;     // per warp: 64 column sums and 64 sums of squares (doubles)
  return s;
}
// Episode statistics accumulate in per-thread columns (n, sum ret, sum ret^2, sum len as doubles; four extrema
// as floats).  A thread touches its column only when one of its episodes ends, so in this kernel the columns
// live in a caller-provided global scratch buffer instead of shared memory (which the weight images need).
__host__ __device__ inline size_t collect_scratch_per_cta(int threads) { return (size_t)threads * (4 * 8 + 4 * 4); }

template <int TASK, int PHYS, bool X3>
__global__ void __launch_bounds__(512, 1) k_collect(const __grid_constant__ KArgs<float> a, const __grid_constant__ CollectArgs p) {
  typedef float T;
  typedef Model<T, TASK, PHYS, true, PDX_RNG_PHILOX, false> Mo;
  using Cfg = ColCfg<X3>;
  constexpr Layout L = Mo::L;
  constexpr int E = Mo::E, QH = Mo::QH;
  constexpr uint32_t R0 = Cfg::kR0, R1 = Cfg::kR1, R2 = Cfg::kR2;
  const DevCfg<T>& c = a.c;
  const int64_t n = a.b.n_envs;
  const int B = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = c.obs_dim, H = c.history, K1 = p.k1, Tn = p.n_steps;
  const int tile = warp >> 2, wq = warp & 3;                  // tile of this warp, its TMEM lane quarter
  const int tile_warps = min(4, (B >> 5) - 4 * tile);         // the last tile of a CTA may be partial
  const int tile_threads = 32 * tile_warps;
  const int bar_id = 1 + tile;                                // named barrier of the tile (0 = __syncthreads)
  const bool leader_warp = wq == 0;
  // Every warp of a tile waits at its hand-off barriers, although only the issuing warp needs the other warps' data:
  // the barriers keep the tile's warps on the same instructions, and the loop body (159 KB of SASS) lives or dies by
  // instruction-cache sharing (leader-only waits and a counter release of the slot measured slower, DESIGN.md §4)

  extern __shared__ __align__(128) unsigned char smem[];
  const ColSmem sp = collect_smem<X3>(K1, D, B >> 5);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem);          // [0] weights, [1 + 2 s] layer 1 of slot s, [2 + 2 s] layer 2
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + 64);
  uint32_t* slot_busy = reinterpret_cast<uint32_t*>(smem + 72);    // [kSlots]
  uint32_t* slot_phase = reinterpret_cast<uint32_t*>(smem + 80);   // [kSlots] parity of the slot's two mbarriers
  uint32_t* tile_info = reinterpret_cast<uint32_t*>(smem + 96);    // [4] slot | parity << 8 of the tile's current policy step
  uint32_t* tile_done = reinterpret_cast<uint32_t*>(smem + 112);   // [4] read by nothing: see the slot release
  float* act_std = reinterpret_cast<float*>(smem + 128);           // exp(log_std)[4], log_std[4]
  float2* norm = reinterpret_cast<float2*>(smem + sp.norm);        // [K1] (mean, 1 / (std + eps))
  float* common = reinterpret_cast<float*>(smem + sp.common);      // w3a[64][4], w3c[64], b3[16]
  float* bw = reinterpret_cast<float*>(smem + sp.weights);         // B1, B2a, B2c (hi) [, the same (lo)]
  unsigned char* xbuf = smem + sp.x;
  T* tile0 = reinterpret_cast<T*>(smem + sp.tiles);
  double* mom = reinterpret_cast<double*>(smem + sp.moments) + (size_t)warp * 128;   // this warp's [2][64] column moments
  double* acc_sum = reinterpret_cast<double*>(p.scratch + (size_t)blockIdx.x * collect_scratch_per_cta(B));
  T* acc_ext = reinterpret_cast<T*>(acc_sum + 4 * B);
  const uint32_t bar_w = smem_u32(mbar);
  const int64_t wwords = collect_w_words(K1);
  const uint32_t x_slot_bytes = (uint32_t)(Cfg::kImages * (K1 / 4) * kLboA);

  // ---- one-time setup
  if (warp == 0) tmem_alloc<512>(smem_u32(tmem_holder));
  if (tid == 0) {                                            // (a CTA may be a single warp)
    mbar_init(bar_w, 1);
    for (int s = 0; s < 2 * Cfg::kSlots; ++s) mbar_init(bar_w + 8 + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int s = 0; s < Cfg::kSlots; ++s) { slot_busy[s] = 0; slot_phase[s] = 0; }
    for (int s = 0; s < 4; ++s) tile_done[s] = 0;
  }
  if (tid < 4) {
    const float ls = tid < p.act_dim ? p.log_std[tid] : 0.0f;
    act_std[tid] = expf(ls);
    act_std[4 + tid] = ls;
  }
  for (int k = tid; k < K1; k += B) {
    float mu = 0.0f, inv = 1.0f;
    if (k < D && p.std) { mu = p.mean[k]; inv = 1.0f / (p.std[k] + p.eps); }
    norm[k] = make_float2(mu, inv);
  }
  // K padding chunks of the operand buffers: zero, once
  {
    const int n_chunks = (D + 3) >> 2;
    for (int e = tid; e < Cfg::kSlots * Cfg::kImages * kTile * (K1 / 4 - n_chunks); e += B) {
      const int m = e & (kTile - 1), r = e >> 7;
      const int kc = n_chunks + r % (K1 / 4 - n_chunks), img = r / (K1 / 4 - n_chunks);
      // (img: slot-major, hi image first; the constant-1 column D starts a padding chunk when D is a multiple of 4)
      const float one = (4 * kc == D && (!X3 || (img & 1) == 0)) ? 1.0f : 0.0f;
      *reinterpret_cast<float4*>(xbuf + (size_t)img * (K1 / 4) * kLboA + kc * kLboA + m * 16) = make_float4(one, 0.f, 0.f, 0.f);
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    acc_sum[k * B + tid] = 0.0;
    acc_ext[k * B + tid] = (k & 1) ? T(-1e30) : T(1e30);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) mom[lane + 32 * k] = 0.0;
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_holder;
  if (tid == 0) {                                            // weight image: common + B1/B2a/B2c (hi) [, (lo)]
    const uint32_t bytes_hi = (uint32_t)((kCommonWords + wwords) * 4), bytes_lo = (uint32_t)(wwords * 4);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_w), "r"(bytes_hi + (X3 ? bytes_lo : 0u)) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(common)),
                 "l"(p.packed), "r"(bytes_hi), "r"(bar_w)
                 : "memory");
    if (X3)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(bw + wwords)),
                   "l"(p.packed + kCommonWords + tc_b_words(K1)), "r"(bytes_lo), "r"(bar_w)
                   : "memory");
  }
  mbar_wait(bar_w, 0);

  const float* w3a = common;
  const float* w3c = common + 256;
  const float* b3 = common + 320;
  const uint32_t b1_s = smem_u32(bw), b2a_s = b1_s + K1 * kN1 * 4, b2c_s = b2a_s + kB2Words * 4;
  const uint32_t lo_off = (uint32_t)wwords * 4;
  T* state = reinterpret_cast<T*>(a.b.state);
  T* my_row = tile0 + (size_t)tid * D;
  const int row = 32 * wq + lane;                              // this thread's row of the tile = its TMEM lane
  // layer-2 biases ride on a constant-1 hidden unit after the actor's last one (the pack put a 1 into row D of B1
  // there, the actor's bias into that unit's row of B2a and the critic's into Bc): pi_h[0] < 64 is required
  const int EPC = B;                                           // environments per CTA and pass
  const bool row_al8 = (D & 1) == 0;                           // rows start 8-byte aligned (tile base is 16-byte aligned)

  for (int64_t g = blockIdx.x; g < p.groups; g += gridDim.x) {
    const int64_t i = g * EPC + tid;
    const bool valid = i < n;
    Mo m(c);
#pragma unroll
    for (int k = 0; k < Mo::NW; ++k) m.w[k] = T(0);
    if (lane == 0) bulk_wait_read<0>();                        // the tile's last copy of the previous pass
    __syncwarp();
    if (valid) {
      m.load(state, n, i);
      const T* o0 = p.obs0 + i * D;                            // the row the rollout starts from = "previous row" of step 0
      for (int k = 0; k < D; ++k) my_row[k] = o0[k];
    }
    StepCtx<T> sc;
    sc.state = state; sc.n = n; sc.i = i; sc.valid = valid; sc.lane = lane; sc.tid = tid; sc.B = B;
    sc.row0 = my_row; sc.row1 = my_row; sc.stg = nullptr; sc.RS = D; sc.acc_sum = acc_sum; sc.acc_ext = acc_ext; sc.NT = 1;
    sc.fast2 = false; sc.latency = Mo::BULLET && c.use_latency; sc.any_fin = false;
    sc.bulk = ((reinterpret_cast<uintptr_t>(a.b.obs) | (uintptr_t)((uint64_t)n * D * sizeof(T))) & 15u) == 0 &&
              (((uint64_t)max((int64_t)0, min((int64_t)32, n - (i - lane))) * D * sizeof(T)) & 15u) == 0;
    const uint64_t ig = (uint64_t)(a.b.env_offset + i);        // global index: policy noise does not depend on the sharding

    for (int t = 0; t <= Tn; ++t) {
      // =========================== policy step of this tile ===========================
      if (leader_warp && lane == 0) {                          // take a slot
        int s = -1;
        for (uint32_t it = 0; s < 0; ++it) {
#pragma unroll
          for (int q = 0; q < Cfg::kSlots; ++q)
            if (s < 0 && atomicCAS(&slot_busy[q], 0u, 1u) == 0u) s = q;
          if (s < 0) { __nanosleep(kSlotSpinNs); if (it > (1u << 24)) __trap(); }
        }
        __threadfence_block();
        tile_info[tile] = (uint32_t)s | (slot_phase[s] << 8);
      }
      named_bar_sync(bar_id, tile_threads);
      const uint32_t info = tile_info[tile];
      const int slot = (int)(info & 0xffu);
      const uint32_t par = info >> 8;
      const uint32_t tcol = tbase + (uint32_t)(slot * Cfg::kSlotCols);
      const uint32_t taddr = tcol + ((uint32_t)(32 * wq) << 16);
      const uint32_t bar1 = bar_w + 8 + 16 * slot, bar2 = bar1 + 8;
      unsigned char* xh = xbuf + (size_t)slot * x_slot_bytes;
      unsigned char* xl = xh + (size_t)(K1 / 4) * kLboA;
      tc_fence_after();
      // ---- X: this thread's standardised row in the canonical K-major layout (row m, K chunk kc at kc * LBO + m * 16)
      // (rows of environments past the end of the shard hold whatever the tile held: rows are independent)
#pragma unroll 3
      for (int kc = 0; kc < (D >> 2); ++kc) {                  // whole chunks
        uint32_t hi[4];
        float lo[4];
        // (normaliser pairs as two 128-bit loads; the row as two 64-bit loads when its start is 8-byte aligned)
        const float4 n01 = reinterpret_cast<const float4*>(norm)[2 * kc], n23 = reinterpret_cast<const float4*>(norm)[2 * kc + 1];
        const float nmx[4] = {n01.x, n01.z, n23.x, n23.z}, nmy[4] = {n01.y, n01.w, n23.y, n23.w};
        float o[4];
        if (row_al8) {
          const float2 a01 = reinterpret_cast<const float2*>(my_row)[2 * kc], a23 = reinterpret_cast<const float2*>(my_row)[2 * kc + 1];
          o[0] = a01.x; o[1] = a01.y; o[2] = a23.x; o[3] = a23.y;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) o[j] = my_row[4 * kc + j];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float x = (o[j] - nmx[j]) * nmy[j];
          hi[j] = X3 ? tf32_rna(x) : __float_as_uint(x);      // single TF32: the tensor core drops the low 13 bits itself
          lo[j] = x - __uint_as_float(hi[j]);
        }
        *reinterpret_cast<uint4*>(xh + kc * kLboA + row * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (X3) *reinterpret_cast<float4*>(xl + kc * kLboA + row * 16) = make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
      if (D & 3) {                                             // the last chunk: data, the constant-1 column D, zeros
        const int kc = D >> 2;
        uint32_t hi[4];
        float lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 4 * kc + j;
          float x = k == D ? 1.0f : 0.0f;                       // column D: constant 1 (row D of B1 = the layer-1 biases)
          if (k < D) { const float2 nm = norm[k]; x = (my_row[k] - nm.x) * nm.y; }
          hi[j] = X3 ? tf32_rna(x) : __float_as_uint(x);
          lo[j] = x - __uint_as_float(hi[j]);
        }
        *reinterpret_cast<uint4*>(xh + kc * kLboA + row * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (X3) *reinterpret_cast<float4*>(xl + kc * kLboA + row * 16) = make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_async_smem();                                      // generic-proxy writes of X -> visible to the tensor core
      named_bar_sync(bar_id, tile_threads);
      // ---- layer 1: D1[128 x 128] = X . B1 (columns 0..63 actor, 64..127 critic)
      if (leader_warp) {
        constexpr uint32_t idesc = make_idesc(kN1);
        constexpr uint32_t lbo_b = kN1 * 16;
        uint64_t ah = make_desc(smem_u32(xh), kLboA, kSbo), al = make_desc(smem_u32(xl), kLboA, kSbo);
        uint64_t bh = make_desc(b1_s, lbo_b, kSbo), bl = make_desc(b1_s + lo_off, lbo_b, kSbo);
#pragma unroll 1
        for (int ks = 0; ks < K1 / 8; ++ks) {
          if (X3) {
            mma_ss(tcol + R0, al, bh, idesc, ks > 0);
            mma_ss(tcol + R0, ah, bl, idesc, 1);
            mma_ss(tcol + R0, ah, bh, idesc, 1);
          } else {
            mma_ss(tcol + R0, ah, bh, idesc, ks > 0);
          }
          ah += (2 * kLboA) >> 4; al += (2 * kLboA) >> 4; bh += (2 * lbo_b) >> 4; bl += (2 * lbo_b) >> 4;
        }
        tc_commit(bar1);
      }
      // the Gaussian draw does not depend on the networks: under layer 1
      float eps[4], lp = 0.0f;
      {
        policy_normals(p.pol_seed, p.pol_counter + (uint64_t)t, ig, eps);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (k < p.act_dim) lp += -0.5f * eps[k] * eps[k] - act_std[4 + k] - 0.9189385332046727f;
      }
      mbar_wait(bar1, par);
      tc_fence_after();
      // ---- layer-1 epilogue of this thread's row: a2 = act(D1 + b1), back into TMEM in place (TF32 hi [, lo])
#pragma unroll 1
      for (int ch = 0; ch < 8; ++ch) {
        uint32_t r[16], lo[16];
        tmem_ld16(taddr + R0 + 16 * ch, r);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float x = __uint_as_float(r[j]);                // (the bias came in through the constant-1 column of X)
          const float y = ch < 4 ? fmaxf(x, 0.0f) : (X3 ? tanh_fast(x) : tanh_mufu(x));
          r[j] = X3 ? tf32_rna(y) : __float_as_uint(y);       // (single TF32: operand truncation by the hardware, as in
          lo[j] = __float_as_uint(y - __uint_as_float(r[j]));   //  any TF32 GEMM fed with float32 data)
        }
        tmem_st16(taddr + R0 + 16 * ch, r);
        if (X3) tmem_st16(taddr + R2 + 16 * ch, lo);
      }
      tmem_wait_st();
      tc_fence_before();
      named_bar_sync(bar_id, tile_threads);
      // ---- layer 2: D2[:, 0:64] = a2[:, 0:64] . B2a, D2[:, 64:128] = a2[:, 64:128] . B2c (A from TMEM)
      if (leader_warp) {
        tc_fence_after();
        constexpr uint32_t idesc = make_idesc(64);
        constexpr uint32_t lbo_b = 64 * 16;
        constexpr uint64_t kstep = (2 * lbo_b) >> 4;
        uint64_t bha = make_desc(b2a_s, lbo_b, kSbo), bhc = make_desc(b2c_s, lbo_b, kSbo);
        uint64_t bla = make_desc(b2a_s + lo_off, lbo_b, kSbo), blc = make_desc(b2c_s + lo_off, lbo_b, kSbo);
        uint32_t a_hi = tcol + R0, a_lo = tcol + R2;
#pragma unroll 1
        for (int ks = 0; ks < 8; ++ks) {
          if (X3) {
            mma_ts(tcol + R1, a_lo, bha, idesc, ks > 0);
            mma_ts(tcol + R1 + 64, a_lo + 64, bhc, idesc, ks > 0);
            mma_ts(tcol + R1, a_hi, bla, idesc, 1);
            mma_ts(tcol + R1 + 64, a_hi + 64, blc, idesc, 1);
            mma_ts(tcol + R1, a_hi, bha, idesc, 1);
            mma_ts(tcol + R1 + 64, a_hi + 64, bhc, idesc, 1);
          } else {
            mma_ts(tcol + R1, a_hi, bha, idesc, ks > 0);
            mma_ts(tcol + R1 + 64, a_hi + 64, bhc, idesc, ks > 0);
          }
          a_hi += 8; a_lo += 8; bha += kstep; bhc += kstep; bla += kstep; blc += kstep;
        }
        {                                                      // critic bias: the actor's constant-1 unit times Bc
          const uint32_t off = (uint32_t)(p.pi_h[0] & ~7);
          if (X3) mma_ts(tcol + R1 + 64, tcol + R0 + off, blc, idesc, 1);     // (the unit's lo part is 0)
          mma_ts(tcol + R1 + 64, tcol + R0 + off, bhc, idesc, 1);
        }
        tc_commit(bar2);
      }
      mbar_wait(bar2, par);
      tc_fence_after();
      // ---- layer-2 epilogue + layer 3 (64 x 4 + 64 x 1 weights, float32 on the CUDA cores)
      float mu[4] = {b3[0], b3[1], b3[2], b3[3]};
      float v = b3[4];
#pragma unroll 1
      for (int ch = 0; ch < 8; ++ch) {
        uint32_t r[16];
        tmem_ld16(taddr + R1 + 16 * ch, r);
        tmem_wait_ld();
        if (ch < 4) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float y = fmaxf(__uint_as_float(r[j]), 0.0f);
            const float4 wv = *reinterpret_cast<const float4*>(w3a + 4 * (16 * ch + j));
            mu[0] = fmaf(y, wv.x, mu[0]); mu[1] = fmaf(y, wv.y, mu[1]); mu[2] = fmaf(y, wv.z, mu[2]); mu[3] = fmaf(y, wv.w, mu[3]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float x = __uint_as_float(r[j]);
            const float y = X3 ? tanh_fast(x) : tanh_mufu(x);
            v = fmaf(y, w3c[16 * (ch - 4) + j], v);
          }
        }
      }
      tc_fence_before();
      named_bar_sync(bar_id, tile_threads);
      if (leader_warp && lane == 0) {                          // every warp of the tile has read its D2 rows: slot back
        // tile_done has no reader.  Its two stores stay because without them ptxas allocates the loop's registers
        // differently, and k_collect measured 0.8 % (single TF32) and 1.2 % (split TF32) slower on a B200 (1,000 W).
        tile_done[tile] = 0u;
        slot_phase[slot] = par ^ 1u;
        __threadfence_block();
        atomicExch(&slot_busy[slot], 0u);
      }
      // ---- outputs of the policy step
      float av[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (k < p.act_dim) av[k] = fmaf(act_std[k], eps[k], mu[k]);
      if (t == Tn) {
        if (valid) p.last_val[i] = v;
        break;
      }
      if (valid) {
        const int64_t o = (int64_t)t * n + i;
        reinterpret_cast<float4*>(p.act)[o] = make_float4(av[0], av[1], av[2], av[3]);
        p.val[o] = v;
        p.logp[o] = lp;
      }
      // ---- running-statistics sums of the policy inputs (OnlineMeanStd.update,
      // utils/online_mean_std.py:70-84, is fed with the T x n observations the policy saw): each lane sums its
      // columns over the warp's 32 rows; the sums are kept about the normaliser's mean
      if (p.obs_moments) {                                      // (the slot is free again: off the tiles' critical path)
        const int rows_w = (int)max((int64_t)0, min((int64_t)32, n - (i - lane)));
        const T* wrow = my_row - lane * D;
        // float32 sums about the warp's own first row (tiny differences for a nearly constant column: no
        // cancellation), moved to the common shift in float64.  Columns 0..31: one lane each over the warp's
        // rows; columns 32..D-1 (two for the 34-wide hover row): nc lanes x G row groups, folded by shuffles
        const int nc = D > 32 ? D - 32 : 0;
        int G = 1;
        while (nc && 2 * G * nc <= 32) G *= 2;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (h == 1 && nc == 0) break;
          const int g = h ? lane / nc : 0, col = h ? 32 + lane % nc : lane, stride = h ? G : 1;
          const bool on = h ? g < G : col < D;
          float cw = 0.0f, s1 = 0.0f, s2 = 0.0f;
          if (on && rows_w > 0) {
            cw = wrow[col];
            for (int r = h ? g : 1; r < rows_w; r += stride) { const float d = wrow[r * D + col] - cw; s1 += d; s2 = fmaf(d, d, s2); }
          }
          if (h)
            for (int sft = G >> 1; sft; sft >>= 1) {
              s1 += __shfl_down_sync(0xffffffffu, s1, sft * nc);
              s2 += __shfl_down_sync(0xffffffffu, s2, sft * nc);
            }
          if (on && g == 0 && rows_w > 0) {
            const double dc = (double)cw - (double)norm[col].x, nr = (double)rows_w;
            mom[col] += (double)s1 + nr * dc;
            mom[64 + col] += (double)s2 + 2.0 * dc * (double)s1 + nr * dc * dc;
          }
        }
      }
      // =========================== env.step of this thread's environment ===========================
      rollout_step<T, TASK, PHYS, true, PDX_RNG_PHILOX, false, 0>(
          a, m, sc, t, make_float4(av[0], av[1], av[2], av[3]), [&](bool pred) { return tile_vote(bar_id, tile_threads, pred); });
    }
    // ---- end of the pass: state and history back
    if (valid) {
      m.store(state, n, i, true);
      store_history<T, E, QH>(state, n, i, L.n_quads, H, [&](int s, int idx) { return my_row[(s + 1) * E + idx]; });
    }
  }
  // any episode finished in any pass of this CTA?  acc_sum[0..B) > 0 tells
  block_reduce_episode_stats(a.b.episode_stats, acc_sum, acc_ext, B, acc_sum[tid] > 0.0);
  if (p.obs_moments) {                                          // (the reduction above contains a block barrier)
    const double* all = reinterpret_cast<const double*>(smem + sp.moments);
    for (int k = tid; k < 2 * D; k += B) {
      const int col = k % D, which = k / D;
      double v = 0.0;
      for (int wv = 0; wv < (B >> 5); ++wv) v += all[(size_t)wv * 128 + 64 * which + col];
      atomicAdd(&p.obs_moments[k], v);
    }
  }
  if (lane == 0) bulk_wait_all();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_free<512>(tbase);
}

template <int TASK, int PHYS, bool X3>
static cudaError_t launch_collect(const KArgs<float>& ka, CollectArgs& p, int sms, cudaStream_t st) {
  // at most 14 warps, and no more than the shared-memory plan admits: wide rows with the split-TF32 images leave
  // room for fewer (D = 40: 10 warps, D = 60: 3) -- the shard then takes more passes
  int max_warps = 14;
  while (max_warps > 1 && collect_smem<X3>(p.k1, ka.c.obs_dim, max_warps).total > kMaxSmemBytes) --max_warps;
  const int64_t n = ka.b.n_envs;
  // passes and warps per CTA: the fewest passes that fit, then the smallest CTA that covers the shard in them
  int64_t passes = (n + (int64_t)sms * max_warps * 32 - 1) / ((int64_t)sms * max_warps * 32);
  int64_t per_cta = (n + (int64_t)sms * passes - 1) / ((int64_t)sms * passes);
  int warps = (int)((per_cta + 31) / 32);
  if (warps < 1) warps = 1;
  if (warps > max_warps) warps = max_warps;
  p.warps_per_cta = warps;
  p.groups = (int32_t)((n + (int64_t)warps * 32 - 1) / ((int64_t)warps * 32));
  const ColSmem sp = collect_smem<X3>(p.k1, ka.c.obs_dim, warps);
  if (sp.total > kMaxSmemBytes) return cudaErrorInvalidConfiguration;
  const cudaError_t e = opt_in_smem(k_collect<TASK, PHYS, X3>, ka.b.device, sp.total);
  if (e != cudaSuccess) return e;
  const unsigned grid = (unsigned)(p.groups < sms ? p.groups : sms);
  k_collect<TASK, PHYS, X3><<<grid, warps * 32, sp.total, st>>>(ka, p);
  return cudaGetLastError();
}

}  // namespace pdx

extern "C" int64_t pdx_collect_scratch_bytes(int32_t device) {
  int sms = 148;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) { cudaGetLastError(); sms = 148; }
  return (int64_t)sms * (int64_t)pdx::collect_scratch_per_cta(512);
}

extern "C" int pdx_collect(const PdxConfig* cfg, const PdxBuffers* buf, const PdxPolicy* pol, const PdxRollout* out,
                           uint64_t seed, uint64_t counter, void* stream) {
  using namespace pdx;
  if (!cfg || !buf || !pol || !out) return set_error(PDX_ERR_INVALID, "pdx_collect: null argument");
  PdxConfig c = *cfg;
  if (pdx_config_finalize(&c)) return PDX_ERR_INVALID;
  if (c.dtype != PDX_DTYPE_F32 || c.rng_mode != PDX_RNG_PHILOX || !c.observation_noise || c.control_mode != PDX_CTRL_PWM ||
      c.task == PDX_TASK_TAKEOFF || (c.obs_dim & 15) == 0 || c.obs_dim > 64 || !c.auto_reset)
    return set_error(PDX_ERR_INVALID, "pdx_collect: supports float32, Philox, observation noise on, PWM control, hover / circle ids, "
                                      "obs_dim <= 64 and not a multiple of 16, auto_reset (use pdx_policy_step_tc + pdx_step otherwise)");
  if (pol->obs_dim != c.obs_dim || (pol->precision != 1 && pol->precision != 3) || !pol->pi || !pol->v || !pol->log_std || !pol->packed)
    return set_error(PDX_ERR_INVALID, "pdx_collect: bad policy description");
  const PdxMlp* pi = pol->pi; const PdxMlp* v = pol->v;
  if (pi->hidden[0] < 1 || pi->hidden[0] > 63 || pi->hidden[1] < 1 || pi->hidden[1] > 64 || pi->n_out < 1 || pi->n_out > 4 ||
      v->hidden[0] < 1 || v->hidden[0] > 64 || v->hidden[1] < 1 || v->hidden[1] > 64 || v->n_out != 1)
    return set_error(PDX_ERR_INVALID, "pdx_collect: networks must have two hidden layers of <= 64 units (actor: first layer <= 63, <= 4 outputs; critic: 1 output)");
  if (out->n_steps < 1 || out->n_steps > (1 << 20) || !out->obs0 || !out->act || !out->val || !out->logp || !out->last_val)
    return set_error(PDX_ERR_INVALID, "pdx_collect: n_steps must be in [1, 2^20] and obs0 / act / val / logp / last_val are required");
  if (!out->scratch || out->scratch_bytes < pdx_collect_scratch_bytes(buf->device))
    return set_error(PDX_ERR_INVALID, "pdx_collect: scratch buffer of pdx_collect_scratch_bytes() bytes required");
  if (buf->n_envs <= 0 || buf->n_envs >= ((int64_t)1 << 31) || !buf->state || !buf->obs || !buf->reward || !buf->cost || !buf->terminated || !buf->truncated)
    return set_error(PDX_ERR_INVALID, "pdx_collect: state / obs / reward / cost / terminated / truncated buffers are required");
  const int rc = select_device(buf->device);
  if (rc) return rc;
  KArgs<float> ka = make_kargs<float>(c, *buf, seed, counter, out->n_steps);
  ka.b.episode_return = nullptr; ka.b.episode_length = nullptr;
  CollectArgs p;
  p.obs_dim = c.obs_dim; p.k1 = tc_k1(c.obs_dim); p.act_dim = pi->n_out; p.n_steps = out->n_steps;
  p.obs0 = out->obs0; p.mean = pol->mean; p.std = pol->std; p.eps = pol->eps; p.log_std = pol->log_std; p.packed = pol->packed;
  for (int k = 0; k < 2; ++k) { p.pi_h[k] = pi->hidden[k]; p.v_h[k] = v->hidden[k]; }
  p.pol_seed = pol->seed; p.pol_counter = pol->counter;
  p.act = out->act; p.val = out->val; p.logp = out->logp; p.last_val = out->last_val;
  p.scratch = reinterpret_cast<unsigned char*>(out->scratch);
  p.obs_moments = out->obs_moments;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, buf->device);
  const bool x3 = pol->precision == 3, bullet = c.physics == PDX_PHYSICS_BULLET, circle = c.task == PDX_TASK_CIRCLE;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
#define PDX_COL(TASK, PHYS) (x3 ? launch_collect<TASK, PHYS, true>(ka, p, sms, st) : launch_collect<TASK, PHYS, false>(ka, p, sms, st))
  if (circle) e = bullet ? PDX_COL(PDX_TASK_CIRCLE, PDX_PHYSICS_BULLET) : PDX_COL(PDX_TASK_CIRCLE, PDX_PHYSICS_SIMPLE);
  else e = bullet ? PDX_COL(PDX_TASK_HOVER, PDX_PHYSICS_BULLET) : PDX_COL(PDX_TASK_HOVER, PDX_PHYSICS_SIMPLE);
#undef PDX_COL
  return cuda_error("pdx_collect", e);
}
