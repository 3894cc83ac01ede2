// Scalar math wrappers (float / double), quaternion helpers and the counter-based RNG.
//
// Quaternion helpers restate the three PyBullet functions the reference's step depends on
// (third-party Bullet3, pybullet.c / btMatrix3x3.h; SURVEY.md Appendix B); call sites in
// the reference: physics.py:160,179, agents.py:446,452, hover.py:146,209,237.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/phoenix_b200.h"

namespace pdx {

template <class T> struct M;

template <> struct M<float> {
  static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
  static __device__ __forceinline__ float fabs(float x) { return fabsf(x); }
  static __device__ __forceinline__ float fmin(float a, float b) { return fminf(a, b); }
  static __device__ __forceinline__ float fmax(float a, float b) { return fmaxf(a, b); }
  static __device__ __forceinline__ float atan2(float y, float x) { return atan2f(y, x); }
  static __device__ __forceinline__ float asin(float x) { return asinf(x); }
  static __device__ __forceinline__ void sincos(float x, float* s, float* c) { sincosf(x, s, c); }
  static __device__ __forceinline__ float floor(float x) { return floorf(x); }
  static __device__ __forceinline__ bool finite(float x) { return isfinite(x); }
  // Box-Muller on two 32-bit words.  Throughput path: uniforms are built with bit operations
  // (no I2F on the XU pipe), log2 / sqrt / sin / cos are single MUFU operations -- noise
  // quality, not trajectory accuracy, is what matters here.
  static __device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float* z0, float* z1) {
    const float u1 = 2.0f - __uint_as_float(0x3f800000u | (a >> 9));     // (0,1]
    const float u2 = __uint_as_float(0x3f800000u | (b >> 9)) - 1.0f;     // [0,1)
    float l2, r, s, c;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * l2));   // -2 ln u1
    const float ang = 6.283185307179586f * u2;
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(ang));
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c) : "f"(ang));
    *z0 = r * c;
    *z1 = r * s;
  }
  static __device__ __forceinline__ float unit(uint32_t a) {             // [0,1)
    return __uint_as_float(0x3f800000u | (a >> 9)) - 1.0f;
  }
  static __device__ __forceinline__ float unit21(uint32_t u) {           // [0,1) from a 21-bit integer
    return __uint_as_float(0x3f800000u | (u << 2)) - 1.0f;
  }
};

template <> struct M<double> {
  static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
  static __device__ __forceinline__ double fabs(double x) { return ::fabs(x); }
  static __device__ __forceinline__ double fmin(double a, double b) { return ::fmin(a, b); }
  static __device__ __forceinline__ double fmax(double a, double b) { return ::fmax(a, b); }
  static __device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
  static __device__ __forceinline__ double asin(double x) { return ::asin(x); }
  static __device__ __forceinline__ void sincos(double x, double* s, double* c) { ::sincos(x, s, c); }
  static __device__ __forceinline__ double floor(double x) { return ::floor(x); }
  static __device__ __forceinline__ bool finite(double x) { return isfinite(x); }
  static __device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, double* z0, double* z1) {
    const double u1 = ((double)a + 0.5) * (1.0 / 4294967296.0);          // (0,1)
    const double u2 = ((double)b + 0.5) * (1.0 / 4294967296.0);
    const double r = ::sqrt(-2.0 * ::log(u1));
    double s, c;
    ::sincos(6.283185307179586476925 * u2, &s, &c);
    *z0 = r * c;
    *z1 = r * s;
  }
  static __device__ __forceinline__ double unit(uint32_t a) {            // [0,1)
    return (double)a * (1.0 / 4294967296.0);
  }
  static __device__ __forceinline__ double unit21(uint32_t u) {          // [0,1) from a 21-bit integer
    return (double)u * (1.0 / 2097152.0);
  }
};

// ---- quaternion helpers ---------------------------------------------------------------------
// pybullet.getQuaternionFromEuler: half-angle products, then normalisation.  q = (x,y,z,w).
template <class T>
__device__ __forceinline__ void quat_from_euler(T roll, T pitch, T yaw, T q[4]) {
  T sphi, cphi, sthe, cthe, spsi, cpsi;
  M<T>::sincos(roll / T(2), &sphi, &cphi);
  M<T>::sincos(pitch / T(2), &sthe, &cthe);
  M<T>::sincos(yaw / T(2), &spsi, &cpsi);
  const T x = sphi * cthe * cpsi - cphi * sthe * spsi;
  const T y = cphi * sthe * cpsi + sphi * cthe * spsi;
  const T z = cphi * cthe * spsi - sphi * sthe * cpsi;
  const T w = cphi * cthe * cpsi + sphi * sthe * spsi;
  const T n = M<T>::sqrt(x * x + y * y + z * z + w * w);
  q[0] = x / n; q[1] = y / n; q[2] = z / n; q[3] = w / n;
}

// pybullet.getMatrixFromQuaternion (btMatrix3x3::setRotation), row-major.
template <class T>
__device__ __forceinline__ void rot_from_quat(const T q[4], T R[9]) {
  const T x = q[0], y = q[1], z = q[2], w = q[3];
  const T s = T(2) / (x * x + y * y + z * z + w * w);
  const T xs = x * s, ys = y * s, zs = z * s;
  const T wx = w * xs, wy = w * ys, wz = w * zs;
  const T xx = x * xs, xy = x * ys, xz = x * zs;
  const T yy = y * ys, yz = y * zs, zz = z * zs;
  R[0] = T(1) - (yy + zz); R[1] = xy - wz;          R[2] = xz + wy;
  R[3] = xy + wz;          R[4] = T(1) - (xx + zz); R[5] = yz - wx;
  R[6] = xz - wy;          R[7] = yz + wx;          R[8] = T(1) - (xx + yy);
}

// pybullet.getEulerFromQuaternion incl. the gimbal-lock branches at |sarg| >= 0.99999.
template <class T>
__device__ __forceinline__ void euler_from_quat(const T q[4], T e[3]) {
  const T x = q[0], y = q[1], z = q[2], w = q[3];
  const T sarg = T(-2) * (x * z - w * y);
  const T half_pi = T(1.5707963267948966192313);
  if (sarg <= T(-0.99999)) {
    e[0] = T(0); e[1] = -half_pi; e[2] = T(2) * M<T>::atan2(x, -y);
  } else if (sarg >= T(0.99999)) {
    e[0] = T(0); e[1] = half_pi; e[2] = T(2) * M<T>::atan2(-x, y);
  } else {
    e[0] = M<T>::atan2(T(2) * (y * z + w * x), w * w - x * x - y * y + z * z);
    e[1] = M<T>::asin(sarg);
    e[2] = M<T>::atan2(T(2) * (x * y + w * z), w * w + x * x - y * y - z * z);
  }
}

// ---- Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3") ------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}

// The policy's action noise: four standard normals for (seed, counter, env), from one Philox call on the counter
// (env_lo, counter, env_hi, "POL") and two float32 Box-Muller pairs.  k_policy, k_policy_tc and k_collect all draw
// it here, so they sample identical actions for the same (seed, counter, env).
__device__ __forceinline__ void policy_normals(uint64_t seed, uint64_t counter, uint64_t env, float eps[4]) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)counter, (uint32_t)(env >> 32), 0x504F4Cu),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  M<float>::box_muller(r.x, r.y, &eps[0], &eps[1]);
  M<float>::box_muller(r.z, r.w, &eps[2], &eps[3]);
}

// Draw-site ids (4th counter word).  One Philox call per site id yields 4 words; a draw block
// of K variates occupies ceil(K/4) consecutive ids.
enum DrawSite : uint32_t {
  SITE_SUBSTEP = 0,      // + 8*substep : +0..2  OU(4n) + gyro bias (3n) + gyro white noise (3n)
  SITE_FINAL_OBS = 64,   // +0..3 normals: pos(3) vel(3) gyro bias(3) gyro white(3) theta(3); +4 uniforms: pos(3) theta(3) (21 bits each)
  SITE_RESET = 80,       // +0..3 task uniforms (<=14), +4..6 motor x / ring rows normals (4+8)
  SITE_DR = 88,          // +0..3 dt,m,Jx,Jy,Jz,ftf0,ftf1, motor T(4), T2W(4) uniforms
  SITE_RESET_OBS1 = 96,  // like SITE_FINAL_OBS
  SITE_RESET_OBS2 = 104,
  SITE_INIT = 112,       // constructor observation call: gyro bias (3n)
};

// Per-thread RNG context.
//  PDX_RNG_PHILOX: counter = (env_lo, counter_lo, env_hi ^ counter_hi<<8, draw site), key = seed.
//  PDX_RNG_TAPE  : parity/debug kernels.  Standardised draws come from a [slots][n_envs]
//                  double tape in the reference's draw order; or, when `dump` is set, Philox
//                  draws are generated as in production and copied out in tape layout
//                  (pdx_dump_draws) so the oracle can replay exactly what the kernel used.
template <class T, int MODE>
struct Rng {
  uint2 key;
  uint32_t env_lo, env_hi, ctr_lo;
  const double* tape;     // column of this env in the current phase's tape
  double* dump;           // TAPE mode only
  int64_t stride;         // n_envs

  static constexpr bool kTape = MODE == PDX_RNG_TAPE;
  __device__ __forceinline__ bool dumping() const { return MODE == PDX_RNG_TAPE && dump != nullptr; }
  __device__ __forceinline__ void dump_value(int slot, double v) const { if (dumping()) dump[(int64_t)slot * stride] = v; }

  __device__ __forceinline__ uint4 raw(uint32_t site) const {
    return philox4x32_10(make_uint4(env_lo, ctr_lo, env_hi, site), key);
  }
  // K standard normals / unit uniforms from ceil(K/4) consecutive draw sites starting at
  // `site0` (Box-Muller pairs words (2j, 2j+1) of the concatenated raw stream).
  template <int K>
  __device__ __forceinline__ void philox_normals(uint32_t site0, T* out) const {
#pragma unroll
    for (int c = 0; c < (K + 3) / 4; ++c) {
      const uint4 r = raw(site0 + c);
      T z[4];
      M<T>::box_muller(r.x, r.y, &z[0], &z[1]);
      if (4 * c + 2 < K) M<T>::box_muller(r.z, r.w, &z[2], &z[3]);
#pragma unroll
      for (int k = 0; k < 4; ++k) if (4 * c + k < K) out[4 * c + k] = z[k];
    }
  }
  template <int K>
  __device__ __forceinline__ void philox_uniforms(uint32_t site0, T* out) const {
#pragma unroll
    for (int c = 0; c < (K + 3) / 4; ++c) {
      const uint4 r = raw(site0 + c);
      const uint32_t v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) if (4 * c + k < K) out[4 * c + k] = M<T>::unit(v[k]);
    }
  }
  // Six unit uniforms from ONE call: 21 bits each (the high 21 bits of the four words, and the low 11 + 10 bits of
  // two word pairs).  The float32 path keeps 23 bits of a word anyway; the sensor model's uniform terms are +-1 mm and
  // +-0.05 degrees wide.  Saves one of the six Philox calls of an observation.
  __device__ __forceinline__ void gen_uniforms6(uint32_t site, T* out) const {
    const uint4 r = raw(site);
    out[0] = M<T>::unit21(r.x >> 11);
    out[1] = M<T>::unit21(r.y >> 11);
    out[2] = M<T>::unit21(r.z >> 11);
    out[3] = M<T>::unit21(r.w >> 11);
    out[4] = M<T>::unit21(((r.x & 0x7FFu) << 10) | (r.y & 0x3FFu));
    out[5] = M<T>::unit21(((r.z & 0x7FFu) << 10) | (r.w & 0x3FFu));
  }
  // Raw generation (no tape, no dump): what the production path consumes.
  template <int K> __device__ __forceinline__ void gen_normals(uint32_t site0, T* out) const { philox_normals<K>(site0, out); }
  template <int K> __device__ __forceinline__ void gen_uniforms(uint32_t site0, T* out) const { philox_uniforms<K>(site0, out); }
  // true when the draws must be the reference's own (recorded) ones, one per reference draw
  __device__ __forceinline__ bool exact_draws() const { return MODE == PDX_RNG_TAPE && dump == nullptr; }
  // Tape slot of draw k: slot0 + k, or slot0 + rel[k] when the reference interleaves other draws.
  template <int K>
  __device__ __forceinline__ void normals_at(uint32_t site0, int slot0, const int (&rel)[K], T* out) const {
    if (MODE == PDX_RNG_TAPE) {
      if (dump) {
        philox_normals<K>(site0, out);
#pragma unroll
        for (int k = 0; k < K; ++k) dump[(int64_t)(slot0 + rel[k]) * stride] = (double)out[k];
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) out[k] = (T)tape[(int64_t)(slot0 + rel[k]) * stride];
      }
    } else {
      philox_normals<K>(site0, out);
    }
  }
  template <int K>
  __device__ __forceinline__ void uniforms_at(uint32_t site0, int slot0, const int (&rel)[K], T* out) const {
    if (MODE == PDX_RNG_TAPE) {
      if (dump) {
        philox_uniforms<K>(site0, out);
#pragma unroll
        for (int k = 0; k < K; ++k) dump[(int64_t)(slot0 + rel[k]) * stride] = (double)out[k];
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) out[k] = (T)tape[(int64_t)(slot0 + rel[k]) * stride];
      }
    } else {
      philox_uniforms<K>(site0, out);
    }
  }
  template <int K>
  __device__ __forceinline__ void normals(uint32_t site0, int slot0, T* out) const {
    int rel[K];
#pragma unroll
    for (int k = 0; k < K; ++k) rel[k] = k;
    normals_at<K>(site0, slot0, rel, out);
  }
  template <int K>
  __device__ __forceinline__ void uniforms(uint32_t site0, int slot0, T* out) const {
    int rel[K];
#pragma unroll
    for (int k = 0; k < K; ++k) rel[k] = k;
    uniforms_at<K>(site0, slot0, rel, out);
  }
};

}  // namespace pdx
