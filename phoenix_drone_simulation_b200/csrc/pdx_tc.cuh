// tcgen05 / TMEM / TMA building blocks shared by the tensor-core policy kernel (pdx_policy_tc.cu) and the fused
// collector kernel (pdx_collect.cu): PTX wrappers, the canonical no-swizzle K-major operand layout, TF32
// rounding and the layout of the packed weight image (written by k_pack_tc in pdx_policy_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace {

constexpr int kTile = 128;         // environments per tile = TMEM lanes = MMA M
constexpr int kN1 = 128;           // actor 64 | critic 64
constexpr int kB2Words = 64 * 64;
constexpr int kBiasTileWords = 8 * (kN1 + 64 + 64);     // K = 8 bias tiles (row k = 0 carries the bias)
constexpr int kCommonWords = 64 * 4 + 64 + 16;          // float32 layer 3: w3a[64][4], w3c[64], b3[16]
constexpr uint32_t kLboA = 2048 + 16;   // bytes between K chunks of the X tile (+16: bank spread for the 128-bit stores)
constexpr uint32_t kSbo = 128;          // bytes between 8-row groups: core matrices are packed
constexpr uint32_t kOnesBytes = 2 * 2048;


// ---------------------------------------------------------------------------------------------
//  PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes (or the hint
// expires) instead of returning at once -- a bare try_wait loop spins, and the spinning warps take issue
// slots and shared-memory pipe bandwidth from the warps that work (37 % of all instructions, measured)
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
  return ok != 0;
}
// bounded: a tensor-core operation that never completes (a malformed descriptor) must not hang the GPU
__device__ __forceinline__ void mbar_wait_thread(uint32_t bar, uint32_t parity) {
  for (uint32_t it = 0; !mbar_try(bar, parity); ++it)
    if (it > (1u << 20)) __trap();
}
// warp-level wait: ONE lane polls (32 lanes hitting the same mbarrier word serialise), the warp
// re-converges on __syncwarp, which also orders the other lanes' later reads after the acquire
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if ((threadIdx.x & 31) == 0) mbar_wait_thread(bar, parity);
  __syncwarp();
}
__device__ __forceinline__ void named_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_free(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {            // warp-uniform call, elected lane commits
  asm volatile(
      "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" ::"r"(bar)
      : "memory");
}

// shared-memory matrix descriptor, no swizzle, K-major canonical layout:
//   element (row, k) of a 4-byte type lives at  (k / 4) * LBO + (row / 8) * SBO + (row % 8) * 16 + (k % 4) * 4
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// instruction descriptor, kind::tf32: D = f32, A = B = tf32, both K-major, M = 128
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTile >> 4) << 24);
}

// Called by ALL lanes of the issuing warp with warp-uniform operands (they then live in uniform registers);
// elect.sync picks one lane and only the tcgen05 instruction itself is predicated on it.
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}

// 32 lanes x 32 bit x 16 columns: thread l of the warp gets columns [c, c+16) of lane (base lane + l)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// round to nearest (ties away) onto the 10 explicit mantissa bits of tf32: two integer operations
// (cvt.rna.tf32.f32 expands to an eight-instruction sequence with special-value handling)
__device__ __forceinline__ uint32_t tf32_rna(float x) { return (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u; }
__device__ __forceinline__ float tanh_mufu(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// tanh(x) = 1 - 2 / (2^(2 log2(e) x) + 1): FMUL, MUFU.EX2, FADD, MUFU.RCP, FFMA; saturates correctly
// (ex2 -> inf gives rcp -> 0) so no clamp is needed; ~1e-6 absolute error
__device__ __forceinline__ float tanh_fast(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(2.885390081777927f * x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}

// K of layer 1: the observation columns, ONE constant-1 column (column D: row D of B1 carries the layer-1 biases, so
// the fused collector needs no bias pass; k_policy_tc keeps that column at 0 and uses its bias tiles), zero padding to
// a multiple of the tf32 MMA K (8).  Rows that are a multiple of 16 wide get no such column: pdx_collect does not take
// them (its bulk-copy rule), and for k_policy_tc alone the extra K step would be wasted shared memory
__host__ __device__ inline int tc_k1(int obs_dim) { return (obs_dim & 15) == 0 ? obs_dim : (obs_dim + 8) & ~7; }
constexpr int kColBiasWords = 8 * 64;                   // K = 8 tile of the collector: row (pi_h1 & 7) = critic layer-2 bias

// floats of one operand image (hi or lo): B1[K1/4][128][4], B2a[16][64][4], B2c[16][64][4], collector bias tile, bias tiles
__host__ __device__ inline int64_t tc_b_words(int k1) { return (int64_t)k1 * kN1 + 2 * kB2Words + kColBiasWords + kBiasTileWords; }

}  // namespace
