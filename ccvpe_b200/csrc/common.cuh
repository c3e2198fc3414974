// Shared helpers for libccvpe_b200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/ccvpe_b200.h"

namespace ccvpe {

// ---- error reporting -------------------------------------------------------------------------------------------
char* last_error_buffer();          // thread-local, 512 bytes
std::atomic<int64_t>& launch_counter();   // process wide

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buffer(), 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CCVPE_REQUIRE(cond, ...)                                           \
  do {                                                                     \
    if (!(cond)) return ::ccvpe::fail(CCVPE_ERR_BAD_ARGUMENT, __VA_ARGS__); \
  } while (0)

inline int check_launch(const char* what) {
  launch_counter().fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(CCVPE_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return CCVPE_OK;
}

#define CCVPE_LAUNCH_CHECK(what)                \
  do {                                          \
    int _rc = ::ccvpe::check_launch(what);      \
    if (_rc != CCVPE_OK) return _rc;            \
  } while (0)

// Optional output placement of the 1x1 SiLU epilogue: pixel (b, h, w) goes to (b, h + lo, w + lo) of a [B, Hp, Wp, ldo]
// image (the pre-zeroed padded staging buffer the depthwise convolution reads).
struct TcOutPad {
  int Hp, Wp, lo;
};

// Arguments of the tensor-core encoder stem (stem_tcgen05.cu); x (planar fp32) or x8 (planar uint8 + the normalisation
// u8 * sc + sh, per-image roll and source row pitch Wsrc) is the image batch.
struct StemTcParams {
  const float* x;
  const uint8_t* x8;
  const int32_t* shift;
  int Wsrc;
  float sc[3], sh[3];
  const float* w;          // fp32 [27][32], k = (ci * 3 + ky) * 3 + kx
  const float* bias;       // fp32 [32]
  __nv_bfloat16* out;      // padded channels-last image [B, Hp, Wp, 32]
  int B, H, W, Ho, Wo, in_lo, out_lo, Hp, Wp, strips, total_tiles;
};
int stem_tcgen05(StemTcParams p, bool circular, bool u8, cudaStream_t st);

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int sm_count();  // cached cudaDevAttrMultiProcessorCount of the current device (148 on B200)

// cudaFuncSetAttribute is per (function, DEVICE): the launchers remember in a per-thread bit mask which devices a kernel's
// attributes were already set on.  Returns true the first time it is called for the calling thread's current device.
inline bool first_use_on_device(uint64_t& mask) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return true;
  const uint64_t bit = 1ull << (dev & 63);
  if (mask & bit) return false;
  mask |= bit;
  return true;
}

// ---- element access ----------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_float(T v);
template <> __device__ __forceinline__ float to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// load 4 consecutive elements as floats (pointer must be 4-element aligned)
__device__ __forceinline__ float4 load4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 load4(const __nv_bfloat16* p) {
  uint2 raw = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 lo = *reinterpret_cast<__nv_bfloat162*>(&raw.x);
  __nv_bfloat162 hi = *reinterpret_cast<__nv_bfloat162*>(&raw.y);
  float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void store4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void store4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 raw;
  raw.x = *reinterpret_cast<uint32_t*>(&lo);
  raw.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = raw;
}

// packed fp32x2 helpers: Blackwell's FFMA2 does two fp32 FMAs per issued instruction, and a bf16x2 word widens to an
// fp32 pair with one shift and one mask
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t bf16x2_to_f32x2(uint32_t v) {
  return pack_f32x2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// a13's orientation rule at a decoded pixel (reference train_VIGOR.py:290-326), evaluated in float64: valid when
// |cos| <= 1 && |sin| <= 1, then degrees(acos(cos)), or for sin < 0 Python's `degrees(-acos(cos)) % 360`; NaN when not
// valid.  pose_finish_kernel and pose_hypotheses_kernel both call it, so a single hypothesis equals decode_pose bit for bit.
__device__ __forceinline__ double pose_angle_deg(float c, float s, bool& ok) {
  ok = fabsf(c) <= 1.f && fabsf(s) <= 1.f;
  double a = __longlong_as_double(0x7ff8000000000000LL);
  if (ok) {
    const double rad2deg = 180.0 / 3.141592653589793238462643383279502884;
    double ac = acos((double)c);
    if (s < 0.f) {
      double r = fmod(-ac * rad2deg, 360.0);  // python's float % : result takes the sign of the divisor
      if (r < 0.0) r += 360.0;
      if (r == 0.0) r = 0.0;
      a = r;
    } else {
      a = ac * rad2deg;
    }
  }
  return a;
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

}  // namespace ccvpe
