// a10 heatmap softmax (models.py:319-320), a12 orientation-field normalisation (models.py:341),
// a13 argmax pose decode (train_VIGOR.py:290-326).  All HBM-bound streaming kernels: 128-bit loads, warp-shuffle
// reductions, every row split over several CTAs so that B rows fill 148 SMs.
#include "common.cuh"

namespace ccvpe {

// ------------------------------------------------------------------------------------------------------------
// softmax over rows of n floats, each row split into `segs` segments
// ------------------------------------------------------------------------------------------------------------
constexpr int kRowThreads = 256;

__host__ __device__ inline int64_t seg_len(int64_t n, int segs) {
  int64_t per = (n + segs - 1) / segs;
  return (per + 3) / 4 * 4;  // keep float4 alignment of segment starts
}

inline int choose_segments(int B, int64_t n) {
  int target = 2 * sm_count();
  int segs = (target + B - 1) / B;
  int64_t max_segs = n / (kRowThreads * 4);  // at least one float4 per thread
  if (max_segs < 1) max_segs = 1;
  if (segs > max_segs) segs = (int)max_segs;
  if (segs > 64) segs = 64;
  if (segs < 1) segs = 1;
  return segs;
}

__global__ void __launch_bounds__(kRowThreads)
softmax_partial_kernel(const float* __restrict__ logits, int64_t n, int segs, float2* __restrict__ partial) {
  const int b = blockIdx.y, sg = blockIdx.x;
  const int64_t len = seg_len(n, segs);
  const int64_t lo = sg * len, hi = min(n, lo + len);
  const float* row = logits + (int64_t)b * n;
  float m = -INFINITY, s = 0.f;
  const bool vec_ok = (n % 4 == 0);
  if (vec_ok) {
    constexpr int U = 4;                                   // independent 16-byte loads in flight per thread
    for (int64_t i0 = lo + threadIdx.x * 4; i0 < hi; i0 += (int64_t)kRowThreads * 4 * U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + (int64_t)u * kRowThreads * 4;
        v[u] = i < hi ? __ldg(reinterpret_cast<const float4*>(row + i))
                      : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      }
      float mx = -INFINITY;
#pragma unroll
      for (int u = 0; u < U; ++u) mx = fmaxf(mx, fmaxf(fmaxf(v[u].x, v[u].y), fmaxf(v[u].z, v[u].w)));
      if (mx > m) {
        s *= expf(m - mx);
        m = mx;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + (int64_t)u * kRowThreads * 4;
        if (i < hi) s += expf(v[u].x - m) + expf(v[u].y - m) + expf(v[u].z - m) + expf(v[u].w - m);
      }
    }
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kRowThreads) {
      float v = row[i];
      if (v > m) {
        s *= expf(m - v);
        m = v;
      }
      s += expf(v - m);
    }
  }
  // block combine
  __shared__ float sm_m[kRowThreads / 32], sm_s[kRowThreads / 32];
  float wm = warp_max(m);
  float ws = warp_sum(m == -INFINITY ? 0.f : s * expf(m - wm));
  if ((threadIdx.x & 31) == 0) {
    sm_m[threadIdx.x >> 5] = wm;
    sm_s[threadIdx.x >> 5] = ws;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    float mm = threadIdx.x < kRowThreads / 32 ? sm_m[threadIdx.x] : -INFINITY;
    float ss = threadIdx.x < kRowThreads / 32 ? sm_s[threadIdx.x] : 0.f;
    float bm = warp_max(mm);
    float bs = warp_sum(mm == -INFINITY ? 0.f : ss * expf(mm - bm));
    if (threadIdx.x == 0) partial[(int64_t)b * segs + sg] = make_float2(bm, bs);
  }
}

__global__ void __launch_bounds__(kRowThreads)
softmax_finish_kernel(const float* __restrict__ logits, float* __restrict__ heat, int64_t n, int segs,
                      const float2* __restrict__ partial) {
  const int b = blockIdx.y, sg = blockIdx.x;
  float M = -INFINITY;
  for (int j = 0; j < segs; ++j) M = fmaxf(M, partial[(int64_t)b * segs + j].x);
  float Z = 0.f;
  for (int j = 0; j < segs; ++j) {
    float2 p = partial[(int64_t)b * segs + j];
    if (p.x != -INFINITY) Z += p.y * expf(p.x - M);
    if (p.y != p.y) Z = p.y;  // NaN somewhere in the row -> whole row NaN (like torch.softmax)
  }
  const float inv = 1.f / Z;
  const int64_t len = seg_len(n, segs);
  const int64_t lo = sg * len, hi = min(n, lo + len);
  const float* row = logits + (int64_t)b * n;
  float* out = heat + (int64_t)b * n;
  if (n % 4 == 0) {
    constexpr int U = 4;
    for (int64_t i0 = lo + threadIdx.x * 4; i0 < hi; i0 += (int64_t)kRowThreads * 4 * U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + (int64_t)u * kRowThreads * 4;
        if (i < hi) v[u] = __ldg(reinterpret_cast<const float4*>(row + i));
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + (int64_t)u * kRowThreads * 4;
        if (i >= hi) break;
        v[u].x = expf(v[u].x - M) * inv;
        v[u].y = expf(v[u].y - M) * inv;
        v[u].z = expf(v[u].z - M) * inv;
        v[u].w = expf(v[u].w - M) * inv;
        __stcs(reinterpret_cast<float4*>(out + i), v[u]);
      }
    }
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kRowThreads) out[i] = expf(row[i] - M) * inv;
  }
}

// ------------------------------------------------------------------------------------------------------------
// orientation field: channels-last (cos, sin) pairs -> unit vectors, planar fp32
// ------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void ori_normalize_kernel(const T* __restrict__ in, int ld, float* __restrict__ out, int64_t HW,
                                     int64_t total) {
  // 4 consecutive pixels per thread: with ld == 2 that is one 32-byte (fp32) / 16-byte (bf16) load and two float4 stores
  const int64_t groups = (total + 3) / 4;
  for (int64_t gidx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; gidx < groups; gidx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i0 = gidx * 4;
    float c[4], s[4];
    const bool fast = (ld == 2) && (i0 + 3 < total) && (HW % 4 == 0);
    if (fast) {
      if constexpr (sizeof(T) == 4) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(in + i0 * 2));
        const float4 b = __ldcs(reinterpret_cast<const float4*>(in + i0 * 2 + 4));
        c[0] = a.x; s[0] = a.y; c[1] = a.z; s[1] = a.w; c[2] = b.x; s[2] = b.y; c[3] = b.z; s[3] = b.w;
      } else {
        const uint4 q = __ldcs(reinterpret_cast<const uint4*>(in + i0 * 2));
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __bfloat1622float2(h[j]);
          c[j] = f.x;
          s[j] = f.y;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t i = i0 + j;
        c[j] = s[j] = 0.f;
        if (i < total) {
          c[j] = to_float(in[i * ld]);
          s[j] = to_float(in[i * ld + 1]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float nrm = fmaxf(sqrtf(c[j] * c[j] + s[j] * s[j]), 1e-12f);
      c[j] /= nrm;
      s[j] /= nrm;
    }
    if (fast) {
      const int64_t b = i0 / HW, p = i0 - b * HW;      // HW % 4 == 0: the 4 pixels share one image
      __stcs(reinterpret_cast<float4*>(out + (b * 2 + 0) * HW + p), make_float4(c[0], c[1], c[2], c[3]));
      __stcs(reinterpret_cast<float4*>(out + (b * 2 + 1) * HW + p), make_float4(s[0], s[1], s[2], s[3]));
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t i = i0 + j;
        if (i < total) {
          const int64_t b = i / HW, p = i - b * HW;
          out[(b * 2 + 0) * HW + p] = c[j];
          out[(b * 2 + 1) * HW + p] = s[j];
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// argmax pose decode
// ------------------------------------------------------------------------------------------------------------
struct ArgPartial {
  float v;
  int is_nan;
  int64_t idx;
};

// numpy argmax semantics: the first NaN wins; otherwise the first occurrence of the maximum
__device__ __forceinline__ bool better(float v, int vn, int64_t vi, float bv, int bn, int64_t bi) {
  if (vn != bn) return vn > bn;
  if (vn) return vi < bi;
  if (v != bv) return v > bv;
  return vi < bi;
}

__device__ __forceinline__ void arg_combine(float& v, int& vn, int64_t& vi, float ov, int on, int64_t oi) {
  if (better(ov, on, oi, v, vn, vi)) {
    v = ov;
    vn = on;
    vi = oi;
  }
}

__device__ void block_arg_reduce(float& v, int& vn, int64_t& vi) {
  __shared__ float sv[kRowThreads / 32];
  __shared__ int sn[kRowThreads / 32];
  __shared__ int64_t si[kRowThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, v, o);
    int on = __shfl_xor_sync(0xffffffffu, vn, o);
    int64_t oi = __shfl_xor_sync(0xffffffffu, vi, o);
    arg_combine(v, vn, vi, ov, on, oi);
  }
  if ((threadIdx.x & 31) == 0) {
    sv[threadIdx.x >> 5] = v;
    sn[threadIdx.x >> 5] = vn;
    si[threadIdx.x >> 5] = vi;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    bool ok = threadIdx.x < (blockDim.x >> 5);
    v = ok ? sv[threadIdx.x] : -INFINITY;
    vn = ok ? sn[threadIdx.x] : 0;
    vi = ok ? si[threadIdx.x] : INT64_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, v, o);
      int on = __shfl_xor_sync(0xffffffffu, vn, o);
      int64_t oi = __shfl_xor_sync(0xffffffffu, vi, o);
      arg_combine(v, vn, vi, ov, on, oi);
    }
  }
}

__global__ void __launch_bounds__(kRowThreads)
argmax_partial_kernel(const float* __restrict__ heat, int64_t n, int segs, ArgPartial* __restrict__ partial) {
  const int b = blockIdx.y, sg = blockIdx.x;
  const int64_t len = seg_len(n, segs);
  const int64_t lo = sg * len, hi = min(n, lo + len);
  const float* row = heat + (int64_t)b * n;
  float v = -INFINITY;
  int vn = 0;
  int64_t vi = INT64_MAX;
  if (n % 4 == 0) {
    for (int64_t i = lo + threadIdx.x * 4; i < hi; i += kRowThreads * 4) {
      float4 q = *reinterpret_cast<const float4*>(row + i);
      float e[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) arg_combine(v, vn, vi, e[j], e[j] != e[j], i + j);
    }
  } else {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kRowThreads) arg_combine(v, vn, vi, row[i], row[i] != row[i], i);
  }
  block_arg_reduce(v, vn, vi);
  if (threadIdx.x == 0) {
    ArgPartial p;
    p.v = v;
    p.is_nan = vn;
    p.idx = vi;
    partial[(int64_t)b * segs + sg] = p;
  }
}

__global__ void pose_finish_kernel(const ArgPartial* __restrict__ partial, int segs, const float* __restrict__ ori,
                                   int64_t n, int W, int64_t* __restrict__ idx, int32_t* __restrict__ rc,
                                   float* __restrict__ cs, double* __restrict__ angle, uint8_t* __restrict__ valid) {
  const int b = blockIdx.x;
  if (threadIdx.x != 0) return;
  float v = -INFINITY;
  int vn = 0;
  int64_t vi = INT64_MAX;
  for (int j = 0; j < segs; ++j) {
    ArgPartial p = partial[(int64_t)b * segs + j];
    arg_combine(v, vn, vi, p.v, p.is_nan, p.idx);
  }
  if (vi == INT64_MAX) vi = 0;  // row of all -inf: numpy returns 0
  idx[b] = vi;
  rc[2 * b + 0] = (int32_t)(vi / W);
  rc[2 * b + 1] = (int32_t)(vi % W);
  float c = ori[((int64_t)b * 2 + 0) * n + vi], s = ori[((int64_t)b * 2 + 1) * n + vi];
  cs[2 * b + 0] = c;
  cs[2 * b + 1] = s;
  bool ok;
  angle[b] = pose_angle_deg(c, s, ok);
  valid[b] = ok ? 1 : 0;
}

}  // namespace ccvpe

extern "C" int64_t ccvpe_softmax_scratch_elems(int B, int64_t n) {
  (void)n;
  return (int64_t)B * 64 * 2;
}

extern "C" int ccvpe_softmax_heatmap(const float* logits, float* heatmap, int B, int64_t n, float* scratch,
                                     void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(logits && heatmap && scratch, "ccvpe_softmax_heatmap: null pointer");
  CCVPE_REQUIRE(B > 0 && n > 0, "ccvpe_softmax_heatmap: bad shape B=%d n=%lld", B, (long long)n);
  CCVPE_REQUIRE(n % 4 != 0 || (aligned16(logits) && aligned16(heatmap)), "ccvpe_softmax_heatmap: misaligned");
  cudaStream_t st = (cudaStream_t)stream;
  int segs = choose_segments(B, n);
  dim3 grid(segs, B);
  softmax_partial_kernel<<<grid, kRowThreads, 0, st>>>(logits, n, segs, (float2*)scratch);
  CCVPE_LAUNCH_CHECK("softmax_partial_kernel");
  softmax_finish_kernel<<<grid, kRowThreads, 0, st>>>(logits, heatmap, n, segs, (const float2*)scratch);
  CCVPE_LAUNCH_CHECK("softmax_finish_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_ori_normalize(const void* in, int dtype, int ld, float* out, int B, int64_t HW, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(in && out, "ccvpe_ori_normalize: null pointer");
  CCVPE_REQUIRE(B > 0 && HW > 0 && ld >= 2 && ld % 2 == 0, "ccvpe_ori_normalize: bad shape B=%d HW=%lld ld=%d", B,
                (long long)HW, ld);
  CCVPE_REQUIRE(dtype == CCVPE_F32 || dtype == CCVPE_BF16, "ccvpe_ori_normalize: bad dtype %d", dtype);
  cudaStream_t st = (cudaStream_t)stream;
  int64_t total = (int64_t)B * HW;
  int blocks = (int)(((total + 3) / 4 + 255) / 256);
  if (blocks > sm_count() * 16) blocks = sm_count() * 16;
  CCVPE_REQUIRE(aligned16(in) && aligned16(out), "ccvpe_ori_normalize: pointers must be 16-byte aligned");
  if (dtype == CCVPE_F32)
    ori_normalize_kernel<float><<<blocks, 256, 0, st>>>((const float*)in, ld, out, HW, total);
  else
    ori_normalize_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)in, ld, out, HW, total);
  CCVPE_LAUNCH_CHECK("ori_normalize_kernel");
  return CCVPE_OK;
}

extern "C" int64_t ccvpe_pose_scratch_bytes(int B, int64_t n) {
  (void)n;
  return (int64_t)B * 64 * (int64_t)sizeof(ccvpe::ArgPartial);
}

extern "C" int ccvpe_pose_decode(const float* heatmap, const float* ori, int B, int H, int W, int64_t* idx, int32_t* rc,
                                 float* cs, double* angle_deg, uint8_t* valid, void* scratch, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(heatmap && ori && idx && rc && cs && angle_deg && valid && scratch, "ccvpe_pose_decode: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0, "ccvpe_pose_decode: bad shape B=%d H=%d W=%d", B, H, W);
  cudaStream_t st = (cudaStream_t)stream;
  int64_t n = (int64_t)H * W;
  CCVPE_REQUIRE(n % 4 != 0 || aligned16(heatmap), "ccvpe_pose_decode: misaligned heatmap");
  int segs = choose_segments(B, n);
  argmax_partial_kernel<<<dim3(segs, B), kRowThreads, 0, st>>>(heatmap, n, segs, (ArgPartial*)scratch);
  CCVPE_LAUNCH_CHECK("argmax_partial_kernel");
  pose_finish_kernel<<<B, 32, 0, st>>>((const ArgPartial*)scratch, segs, ori, n, W, idx, rc, cs, angle_deg, valid);
  CCVPE_LAUNCH_CHECK("pose_finish_kernel");
  return CCVPE_OK;
}
