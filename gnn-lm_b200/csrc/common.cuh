// Shared helpers for libgnnlm_sm100.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gnnlm_sm100.h"

namespace gnnlm {

void set_error(const char* fmt, ...);

#define GNNLM_CHECK_ARG(cond, code, ...) \
  do {                                   \
    if (!(cond)) {                       \
      gnnlm::set_error(__VA_ARGS__);     \
      return (code);                     \
    }                                    \
  } while (0)

// Launch check without synchronising: reports configuration errors only.
#define GNNLM_LAUNCH_CHECK(name)                                              \
  do {                                                                        \
    cudaError_t e__ = cudaGetLastError();                                     \
    if (e__ != cudaSuccess) {                                                 \
      gnnlm::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return (int32_t)e__;                                                    \
    }                                                                         \
  } while (0)

#define GNNLM_CUDA(call)                                                        \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) {                                                   \
      gnnlm::set_error("%s failed: %s", #call, cudaGetErrorString(e__));        \
      return (int32_t)e__;                                                      \
    }                                                                           \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// cudaFuncSetAttribute acts on the current device only, so a one-time set-up is remembered per device (index into a
// [MAX_DEVICES] flag array) -- a process that drives several GPUs configures each of them.
constexpr int MAX_DEVICES = 64;
static inline int device_slot() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) {
    cudaGetLastError();
    d = 0;
  }
  return d < MAX_DEVICES ? d : MAX_DEVICES - 1;
}

__device__ __forceinline__ int64_t live_rows(int64_t cap, const int32_t* dev) {
  if (dev == nullptr) return cap;
  int64_t n = (int64_t)__ldg(dev);
  return n < cap ? n : cap;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- typed row access: load C contiguous elements starting at p (C in {1,2,4,8,16,32}) as fp32 ----
template <int C>
__device__ __forceinline__ void load_f32(const float* __restrict__ p, float (&r)[C]) {
  if constexpr (C % 4 == 0) {
#pragma unroll
    for (int i = 0; i < C / 4; ++i) {
      float4 t = __ldg(reinterpret_cast<const float4*>(p) + i);
      r[4 * i] = t.x; r[4 * i + 1] = t.y; r[4 * i + 2] = t.z; r[4 * i + 3] = t.w;
    }
  } else if constexpr (C == 2) {
    float2 t = __ldg(reinterpret_cast<const float2*>(p));
    r[0] = t.x; r[1] = t.y;
  } else {
#pragma unroll
    for (int i = 0; i < C; ++i) r[i] = __ldg(p + i);
  }
}
template <int C>
__device__ __forceinline__ void load_bf16(const __nv_bfloat16* __restrict__ p, float (&r)[C]) {
  if constexpr (C % 8 == 0) {
#pragma unroll
    for (int i = 0; i < C / 8; ++i) {
      uint4 t = __ldg(reinterpret_cast<const uint4*>(p) + i);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 f = __bfloat1622float2(h[j]);
        r[8 * i + 2 * j] = f.x; r[8 * i + 2 * j + 1] = f.y;
      }
    }
  } else if constexpr (C == 4) {
    uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
    float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
    r[0] = a.x; r[1] = a.y; r[2] = b.x; r[3] = b.y;
  } else {
#pragma unroll
    for (int i = 0; i < C; ++i) r[i] = __bfloat162float(p[i]);
  }
}
template <typename T, int C>
__device__ __forceinline__ void load_row(const T* __restrict__ p, float (&r)[C]) {
  if constexpr (sizeof(T) == 4) load_f32<C>(reinterpret_cast<const float*>(p), r);
  else load_bf16<C>(reinterpret_cast<const __nv_bfloat16*>(p), r);
}
template <int C>
__device__ __forceinline__ void store_f32(float* __restrict__ p, const float (&r)[C]) {
  if constexpr (C % 4 == 0) {
#pragma unroll
    for (int i = 0; i < C / 4; ++i)
      reinterpret_cast<float4*>(p)[i] = make_float4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
  } else if constexpr (C == 2) {
    *reinterpret_cast<float2*>(p) = make_float2(r[0], r[1]);
  } else {
#pragma unroll
    for (int i = 0; i < C; ++i) p[i] = r[i];
  }
}

// ---- split-fp16 (GNNLM_F16X2) helpers: 4 floats <-> (hi, lo) packed fp16 quads ----
__device__ __forceinline__ void split4_f16(float x0, float x1, float x2, float x3, uint2& hi, uint2& lo) {
  x0 = fminf(fmaxf(x0, -65504.f), 65504.f); x1 = fminf(fmaxf(x1, -65504.f), 65504.f);
  x2 = fminf(fmaxf(x2, -65504.f), 65504.f); x3 = fminf(fmaxf(x3, -65504.f), 65504.f);
  const __half2 h01 = __floats2half2_rn(x0, x1), h23 = __floats2half2_rn(x2, x3);
  const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
  const __half2 l01 = __floats2half2_rn(x0 - f01.x, x1 - f01.y), l23 = __floats2half2_rn(x2 - f23.x, x3 - f23.y);
  hi.x = *reinterpret_cast<const uint32_t*>(&h01); hi.y = *reinterpret_cast<const uint32_t*>(&h23);
  lo.x = *reinterpret_cast<const uint32_t*>(&l01); lo.y = *reinterpret_cast<const uint32_t*>(&l23);
}
__device__ __forceinline__ float4 join4_f16(uint2 hi, uint2 lo) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hi.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&hi.y));
  const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&lo.x)), d = __half22float2(*reinterpret_cast<const __half2*>(&lo.y));
  return make_float4(a.x + c.x, a.y + c.y, b.x + d.x, b.y + d.y);
}

// ---- e4m3 companions of a split-fp16 quad (operands of the FP8 correction MMAs of gnnlm_linear_f16f8):
// hi8 = e4m3(hi), lo8 = e4m3(2^10 * lo), round to nearest even, saturating at +-448
__device__ __forceinline__ uint32_t e4m3x4(uint2 v) {
  const __half2_raw a = *reinterpret_cast<const __half2_raw*>(&v.x), b = *reinterpret_cast<const __half2_raw*>(&v.y);
  return (uint32_t)__nv_cvt_halfraw2_to_fp8x2(a, __NV_SATFINITE, __NV_E4M3) |
         ((uint32_t)__nv_cvt_halfraw2_to_fp8x2(b, __NV_SATFINITE, __NV_E4M3) << 16);
}
__device__ __forceinline__ void q8_from_split4(uint2 hi, uint2 lo, uint32_t& hi8, uint32_t& lo8) {
  const __half2 s = __floats2half2_rn(1024.f, 1024.f);
  uint2 ls;
  const __half2 l0 = __hmul2(*reinterpret_cast<const __half2*>(&lo.x), s), l1 = __hmul2(*reinterpret_cast<const __half2*>(&lo.y), s);
  ls.x = *reinterpret_cast<const uint32_t*>(&l0);
  ls.y = *reinterpret_cast<const uint32_t*>(&l1);
  hi8 = e4m3x4(hi);
  lo8 = e4m3x4(ls);
}

// ---- GNNLM_F24: an fp32 value rounded to its top three bytes (sign, 8 exponent bits, 15 mantissa bits: 2^-16 relative), stored
// as a 16-bit plane (bytes 3, 2 -- the value's bf16 truncation) and a byte plane (byte 1) with the SAME row stride in elements, so the
// byte of the element at 16-bit address a sits at a / 2 + bias.  No float conversions either way: byte permutes only.
// The attention inputs Q | K' | V' of the ntgt side in MATH_F16F8 (written by the projection's epilogue, read by cluster_attn.cu):
// 3 bytes per element instead of 4 through HBM, twice.
__device__ __forceinline__ void f24_pack4(float y0, float y1, float y2, float y3, uint2& hi, uint32_t& lo) {
  const uint32_t u0 = __float_as_uint(y0) + 0x80u, u1 = __float_as_uint(y1) + 0x80u, u2 = __float_as_uint(y2) + 0x80u,
                 u3 = __float_as_uint(y3) + 0x80u;                              // round to nearest at bit 8 (sign-magnitude: ties away)
  hi.x = __byte_perm(u0, u1, 0x7632);
  hi.y = __byte_perm(u2, u3, 0x7632);
  lo = __byte_perm(__byte_perm(u0, u1, 0x0051), __byte_perm(u2, u3, 0x0051), 0x5410);
}
// C = 4 features: 8 B of the 16-bit plane + 4 B of the byte plane (byte address = 16-bit address / 2 + bias)
__device__ __forceinline__ void load_row_f24(const __half* __restrict__ p, int64_t bias, float (&r)[4]) {
  const uint2 h = __ldg(reinterpret_cast<const uint2*>(p));
  const uint32_t l = __ldg(reinterpret_cast<const uint32_t*>((int64_t)(reinterpret_cast<uintptr_t>(p) >> 1) + bias));
  r[0] = __uint_as_float(__byte_perm(h.x, l, 0x1040) & 0xffffff00u);
  r[1] = __uint_as_float(__byte_perm(h.x, l, 0x3250) & 0xffffff00u);
  r[2] = __uint_as_float(__byte_perm(h.y, l, 0x1060) & 0xffffff00u);
  r[3] = __uint_as_float(__byte_perm(h.y, l, 0x3270) & 0xffffff00u);
}

}  // namespace gnnlm
