// Backward kernels of the post-encoder path (BASELINE.json configs[4]: the CVM_VIGOR training step; SURVEY section 8(f)-1).
//
//   * weight gradient of the implicit GEMM (CUDA-core fp32 backend; the tcgen05 backend lives in wgrad_tcgen05.cu)
//   * (weighted, bucketed) column sums: bias gradients and the rank-1 "max score" weight of the transposed convs
//   * ReLU mask, planar <-> channels-last helpers for incoming gradients
//   * backward of the orientation-field normalisation (reference models.py:341)
//   * backward of the rolled cosine matching + F.normalize of one level (reference models.py:186-205)
//   * fused forward+backward of the three training losses (reference losses.py:4-29)
//   * backward of the ground descriptor heads (reference models.py:57-97, 152-157)
//
// Data-gradient (dgrad) of the convolutions needs no kernel of its own: the gradient of a 3x3 pad-1 conv is a 3x3 pad-1
// conv with flipped, transposed weights, the gradient of the k2 s2 transposed conv is a k2 s2 conv, and vice versa -- all
// three are `ccvpe_igemm` calls on re-laid-out weights (ccvpe_b200/training.py).
//
// Every reduction here is deterministic: partial sums go to a caller-provided workspace and are combined in a fixed order.
#include <cfloat>
#include <cstring>

#include "common.cuh"

namespace ccvpe {

// ====================================================================================================================
// wgrad (SIMT):  out[tap][c][n] = sum_m A[b, ho*stride + ty - pad, wo*stride + tx - pad, c] * G[m, n] * g_row_scale[m]
// GEMM view: Q = taps * (c0 + c1) rows ("q" = (tap, c)), N columns, K = M pixels.  Tile TQ x TN per CTA, KP pixels per
// shared-memory stage, split-K over pixel ranges (blockIdx.z) with partial tiles in the workspace.
// ====================================================================================================================
constexpr int WG_KP = 32;
constexpr int WG_THREADS = 256;

struct WgradArgs {
  ccvpe_wgrad_desc d;
  int M, Q, ctot, splits, pix_per_split;
  float* dst;   // out (splits == 1) or workspace [splits][Q][N]
};

template <typename T, int TQ, int TN>
__global__ void __launch_bounds__(WG_THREADS) wgrad_simt_kernel(const WgradArgs a) {
  const ccvpe_wgrad_desc& d = a.d;
  constexpr int MQ = TQ / 16, MN = TN / 16;
  constexpr int AQ4 = TQ / 4;                         // float4 groups per A row
  constexpr int A_LOADS = WG_KP * AQ4 / WG_THREADS;   // per thread per stage
  constexpr int GN4 = TN / 4;
  constexpr int G_GROUPS = WG_KP * GN4;               // may be < WG_THREADS
  constexpr int G_LOADS = (G_GROUPS + WG_THREADS - 1) / WG_THREADS;
  __shared__ __align__(16) float As[WG_KP][TQ];
  __shared__ __align__(16) float Gs[WG_KP][TN];

  const int t = threadIdx.x;
  const int tq = t >> 4, tn = t & 15;
  const int q0 = blockIdx.x * TQ, n0 = blockIdx.y * TN;
  const int HWo = d.Hout * d.Wout;
  const int m_begin = blockIdx.z * a.pix_per_split;
  const int m_end = min(a.M, m_begin + a.pix_per_split);

  // the (tap, channel) group this thread stages: fixed for the whole kernel
  const int a_q4 = (t % AQ4) * 4;
  const int a_p0 = t / AQ4;
  const int q = q0 + a_q4;
  const bool q_ok = q < a.Q;
  const int tap = q_ok ? q / a.ctot : 0;
  const int c = q_ok ? q - tap * a.ctot : 0;
  const int ty = tap / d.kw - d.pad, tx = tap % d.kw - d.pad;
  const T* src = static_cast<const T*>(c < d.c0 ? d.a0 : d.a1);
  const int ld = c < d.c0 ? d.ld0 : d.ld1;
  const int cs = c < d.c0 ? c : c - d.c0;
  const T* G = static_cast<const T*>(d.g);

  float acc[MQ][MN];
#pragma unroll
  for (int i = 0; i < MQ; ++i)
#pragma unroll
    for (int j = 0; j < MN; ++j) acc[i][j] = 0.f;

  for (int m0 = m_begin; m0 < m_end; m0 += WG_KP) {
#pragma unroll
    for (int k = 0; k < A_LOADS; ++k) {
      const int p = a_p0 + k * (WG_THREADS / AQ4);
      const int m = m0 + p;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q_ok && m < m_end) {
        const int b = m / HWo, r = m - b * HWo;
        const int ho = r / d.Wout, wo = r - ho * d.Wout;
        const int hi = ho * d.stride + ty, wi = wo * d.stride + tx;
        if (hi >= 0 && hi < d.Hin && wi >= 0 && wi < d.Win)
          v = load4(src + (((int64_t)b * d.Hin + hi) * d.Win + wi) * ld + cs);
      }
      *reinterpret_cast<float4*>(&As[p][a_q4]) = v;
    }
#pragma unroll
    for (int k = 0; k < G_LOADS; ++k) {
      const int gid = t + k * WG_THREADS;
      if (gid < G_GROUPS) {
        const int p = gid / GN4, n4 = (gid % GN4) * 4;
        const int m = m0 + p;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < m_end && n0 + n4 < d.N) {
          v = load4(G + (int64_t)m * d.ldg + n0 + n4);
          if (d.g_row_scale) {
            const float s = __ldg(d.g_row_scale + m);
            v.x *= s; v.y *= s; v.z *= s; v.w *= s;
          }
        }
        *reinterpret_cast<float4*>(&Gs[p][n4]) = v;
      }
    }
    __syncthreads();
#pragma unroll 8
    for (int p = 0; p < WG_KP; ++p) {
      float av[MQ], gv[MN];
#pragma unroll
      for (int i = 0; i < MQ; i += 4) {
        const float4 x = *reinterpret_cast<const float4*>(&As[p][tq * MQ + i]);
        av[i] = x.x; av[i + 1] = x.y; av[i + 2] = x.z; av[i + 3] = x.w;
      }
      if (MN >= 4) {
#pragma unroll
        for (int j = 0; j < MN; j += 4) {
          const float4 x = *reinterpret_cast<const float4*>(&Gs[p][tn * MN + (j & ~3)]);
          gv[j] = x.x;
          if (j + 1 < MN) gv[j + 1] = x.y;
          if (j + 2 < MN) gv[j + 2] = x.z;
          if (j + 3 < MN) gv[j + 3] = x.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < MN; ++j) gv[j] = Gs[p][tn * MN + j];
      }
#pragma unroll
      for (int i = 0; i < MQ; ++i)
#pragma unroll
        for (int j = 0; j < MN; ++j) acc[i][j] = fmaf(av[i], gv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* dst = a.dst + (int64_t)blockIdx.z * a.Q * d.N;
#pragma unroll
  for (int i = 0; i < MQ; ++i) {
    const int qq = q0 + tq * MQ + i;
    if (qq >= a.Q) continue;
#pragma unroll
    for (int j = 0; j < MN; ++j) {
      const int nn = n0 + tn * MN + j;
      if (nn < d.N) dst[(int64_t)qq * d.N + nn] = acc[i][j];
    }
  }
}

// out[e] = sum_{s < splits} ws[s][e], in order (deterministic)
__global__ void reduce_splits_kernel(const float* __restrict__ ws, float* __restrict__ out, int64_t n, int splits) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += ws[(int64_t)k * n + e];
    out[e] = s;
  }
}

// host-side launcher (also used by wgrad_tcgen05.cu: kernels cannot be launched across translation units without -rdc)
int launch_reduce_splits(const float* ws, float* out, int64_t n, int splits, cudaStream_t st) {
  int blocks = (int)((n + 255) / 256);
  if (blocks > 8 * sm_count()) blocks = 8 * sm_count();
  reduce_splits_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, st>>>(ws, out, n, splits);
  return check_launch("reduce_splits_kernel");
}

struct WgradPlan {
  int tq, tn, q_tiles, n_tiles, splits, pix_per_split;
};

static WgradPlan plan_wgrad(const ccvpe_wgrad_desc& d) {
  WgradPlan p;
  const int Q = d.kh * d.kw * (d.c0 + d.c1);
  const int M = d.B * d.Hout * d.Wout;
  p.tn = d.N <= 16 ? 16 : 64;
  p.tq = d.N <= 16 ? 128 : 64;
  p.q_tiles = (Q + p.tq - 1) / p.tq;
  p.n_tiles = (d.N + p.tn - 1) / p.tn;
  const int tiles = p.q_tiles * p.n_tiles;
  int splits = (4 * sm_count() + tiles - 1) / tiles;
  const int max_splits = (M + 4 * WG_KP - 1) / (4 * WG_KP);     // at least 4 stages of pixels per split
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int pps = (M + splits - 1) / splits;
  pps = (pps + WG_KP - 1) / WG_KP * WG_KP;
  p.pix_per_split = pps;
  p.splits = (M + pps - 1) / pps;
  return p;
}

int wgrad_tcgen05_supported(const ccvpe_wgrad_desc& d);                    // wgrad_tcgen05.cu
int64_t wgrad_tcgen05_workspace_elems(const ccvpe_wgrad_desc& d);
int wgrad_tcgen05(const ccvpe_wgrad_desc& d, cudaStream_t st);

static int check_wgrad_desc(const ccvpe_wgrad_desc* d) {
  CCVPE_REQUIRE(d && d->a0 && d->g && d->out, "ccvpe_wgrad: null pointer");
  CCVPE_REQUIRE(d->B > 0 && d->Hin > 0 && d->Win > 0 && d->Hout > 0 && d->Wout > 0 && d->N > 0, "ccvpe_wgrad: bad shape");
  CCVPE_REQUIRE(d->c0 > 0 && d->c0 % 4 == 0 && d->c1 >= 0 && d->c1 % 4 == 0 && d->ld0 >= d->c0 && d->ld0 % 4 == 0 &&
                    (d->c1 == 0 || (d->a1 && d->ld1 >= d->c1 && d->ld1 % 4 == 0)),
                "ccvpe_wgrad: source channels / strides must be multiples of 4 (c0=%d c1=%d ld0=%d ld1=%d)", d->c0, d->c1,
                d->ld0, d->ld1);
  CCVPE_REQUIRE(d->N % 4 == 0 && d->ldg >= d->N && d->ldg % 4 == 0, "ccvpe_wgrad: N=%d / ldg=%d must be multiples of 4", d->N,
                d->ldg);
  CCVPE_REQUIRE(d->kh > 0 && d->kw > 0 && d->kh <= 3 && d->kw <= 3 && d->stride > 0 && d->pad >= 0, "ccvpe_wgrad: bad geometry");
  CCVPE_REQUIRE(d->dtype == CCVPE_F32 || d->dtype == CCVPE_BF16, "ccvpe_wgrad: bad dtype");
  CCVPE_REQUIRE((int64_t)d->B * d->Hout * d->Wout < (1LL << 31), "ccvpe_wgrad: too many pixels");
  return CCVPE_OK;
}

}  // namespace ccvpe

extern "C" int64_t ccvpe_wgrad_workspace_elems(const ccvpe_wgrad_desc* d) {
  using namespace ccvpe;
  if (check_wgrad_desc(d) != CCVPE_OK) return -1;
  const WgradPlan p = plan_wgrad(*d);
  int64_t simt = p.splits > 1 ? (int64_t)p.splits * d->kh * d->kw * (d->c0 + d->c1) * d->N : 0;
  int64_t tc = (d->backend != CCVPE_BACKEND_SIMT && wgrad_tcgen05_supported(*d)) ? wgrad_tcgen05_workspace_elems(*d) : 0;
  return (simt > tc ? simt : tc) + 64;
}

extern "C" int ccvpe_wgrad_plan(const ccvpe_wgrad_desc* d) {
  using namespace ccvpe;
  int rc = check_wgrad_desc(d);
  if (rc != CCVPE_OK) return rc;
  return (d->backend != CCVPE_BACKEND_SIMT && wgrad_tcgen05_supported(*d)) ? 1 : 0;
}

extern "C" int ccvpe_wgrad(const ccvpe_wgrad_desc* d, void* stream) {
  using namespace ccvpe;
  int rc = check_wgrad_desc(d);
  if (rc != CCVPE_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const bool tc_ok = wgrad_tcgen05_supported(*d) != 0;
  if (d->backend == CCVPE_BACKEND_TCGEN05 && !tc_ok)
    return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_wgrad: shape / dtype not supported by the tcgen05 backend");
  if (d->backend != CCVPE_BACKEND_SIMT && tc_ok) return wgrad_tcgen05(*d, st);
  WgradArgs a;
  a.d = *d;
  a.M = d->B * d->Hout * d->Wout;
  a.ctot = d->c0 + d->c1;
  a.Q = d->kh * d->kw * a.ctot;
  const WgradPlan p = plan_wgrad(*d);
  a.splits = p.splits;
  a.pix_per_split = p.pix_per_split;
  const int64_t n_out = (int64_t)a.Q * d->N;
  if (p.splits > 1) {
    CCVPE_REQUIRE(d->workspace && d->workspace_elems >= (int64_t)p.splits * n_out, "ccvpe_wgrad: workspace too small");
    a.dst = d->workspace;
  } else {
    a.dst = d->out;
  }
  const dim3 grid(p.q_tiles, p.n_tiles, p.splits);
#define CCVPE_WG(TT, TQ_, TN_) wgrad_simt_kernel<TT, TQ_, TN_><<<grid, WG_THREADS, 0, st>>>(a)
  if (d->dtype == CCVPE_F32) {
    if (p.tn == 16) CCVPE_WG(float, 128, 16); else CCVPE_WG(float, 64, 64);
  } else {
    if (p.tn == 16) CCVPE_WG(__nv_bfloat16, 128, 16); else CCVPE_WG(__nv_bfloat16, 64, 64);
  }
#undef CCVPE_WG
  CCVPE_LAUNCH_CHECK("wgrad_simt_kernel");
  if (p.splits > 1) {
    int blocks = (int)((n_out + 255) / 256);
    if (blocks > 8 * sm_count()) blocks = 8 * sm_count();
    reduce_splits_kernel<<<blocks, 256, 0, st>>>(d->workspace, d->out, n_out, p.splits);
    CCVPE_LAUNCH_CHECK("reduce_splits_kernel");
  }
  return CCVPE_OK;
}

// ====================================================================================================================
// Bucketed, weighted column sums over a channels-last image:
//   out[(y % s) * s + (x % s)][c] = sum_{b, y, x} w[b, y / s, x / s] * X[b, y, x, c]        (w == NULL: 1;  s in {1, 2})
// s == 1: bias gradient of a conv (sum of dY over pixels).  s == 2 with w = max score map: gradient of the rank-1 weight
// row of a k2 s2 transposed conv (d r1_w[(i, j), co]); s == 2 with w == NULL summed over buckets by the caller: its bias.
// ====================================================================================================================
namespace ccvpe {

constexpr int CS_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(CS_THREADS)
colsum_partial_kernel(const T* __restrict__ x, int64_t n_pix, int H, int W, int C, int ld, const float* __restrict__ w,
                      int s, int pix_per_block, float* __restrict__ ws) {
  // thread layout: groups of 4 channels; lanes = CS_THREADS / (C / 4) pixels in flight (host guarantees C/4 <= 256)
  extern __shared__ float red[];                       // [lanes][buckets * C]
  const int G = C >> 2;
  const int lanes = CS_THREADS / G;
  const int cg = threadIdx.x % G, pl = threadIdx.x / G;
  const int buckets = s * s;
  const int64_t p_lo = (int64_t)blockIdx.x * pix_per_block;
  const int64_t p_hi = min(n_pix, p_lo + pix_per_block);
  float acc[4][4];
#pragma unroll
  for (int k = 0; k < 4; ++k) acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f;
  if (pl < lanes) {
    constexpr int U = 4;                               // independent loads in flight per thread (the loop is latency bound)
    for (int64_t p0 = p_lo + pl; p0 < p_hi; p0 += (int64_t)lanes * U) {
      float4 v[U];
      float wt[U];
      int bucket[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t p = p0 + (int64_t)u * lanes;
        bucket[u] = -1;
        wt[u] = 1.f;
        if (p < p_hi) {
          v[u] = load4(x + p * ld + cg * 4);
          bucket[u] = 0;
          if (s == 2 || w) {
            const uint32_t pp = (uint32_t)p, hw = (uint32_t)(H * W);      // (n_pix < 2^31: checked on the host)
            const uint32_t b = pp / hw, r = pp - b * hw;
            const uint32_t y = r / (uint32_t)W, xx = r - y * (uint32_t)W;
            if (s == 2) bucket[u] = (int)((y & 1u) * 2u + (xx & 1u));
            if (w) wt[u] = __ldg(w + ((int64_t)b * (H / s) + y / s) * (W / s) + xx / s);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k == bucket[u]) {
            acc[k][0] = fmaf(wt[u], v[u].x, acc[k][0]);
            acc[k][1] = fmaf(wt[u], v[u].y, acc[k][1]);
            acc[k][2] = fmaf(wt[u], v[u].z, acc[k][2]);
            acc[k][3] = fmaf(wt[u], v[u].w, acc[k][3]);
          }
        }
      }
    }
    for (int k = 0; k < buckets; ++k)
#pragma unroll
      for (int j = 0; j < 4; ++j) red[((int64_t)pl * buckets + k) * C + cg * 4 + j] = acc[k][j];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < buckets * C; e += CS_THREADS) {
    float sum = 0.f;
    for (int l = 0; l < lanes; ++l) sum += red[(int64_t)l * buckets * C + e];    // fixed order
    ws[(int64_t)blockIdx.x * buckets * C + e] = sum;
  }
}

// out[e] = sum_blocks ws[block][e]: one WARP per output element (lanes stride over the blocks, then a fixed shuffle tree --
// deterministic); the column counts here are tiny, so a thread-per-element loop over ~600 partials would be pure latency
__global__ void colsum_final_kernel(const float* __restrict__ ws, float* __restrict__ out, int n_out, int blocks) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_out) return;
  float s = 0.f;
  for (int k = lane; k < blocks; k += 32) s += ws[(int64_t)k * n_out + warp];
  s = warp_sum(s);
  if (lane == 0) out[warp] = s;
}

}  // namespace ccvpe

extern "C" int64_t ccvpe_colsum_workspace_elems(int64_t n_pix, int C, int s) {
  using namespace ccvpe;
  if (n_pix <= 0 || C <= 0 || (s != 1 && s != 2)) return -1;
  return 4LL * sm_count() * s * s * C + 64 + 4096;      // at most 4 blocks per SM, each one partial row per bucket
}

extern "C" int ccvpe_colsum(const void* x, int dtype, int B, int H, int W, int C, int ld, const float* w, int s,
                            float* out, float* workspace, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && out && workspace, "ccvpe_colsum: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && C % 4 == 0 && ld >= C && ld % 4 == 0,
                "ccvpe_colsum: bad shape C=%d ld=%d", C, ld);
  CCVPE_REQUIRE(s == 1 || (s == 2 && H % 2 == 0 && W % 2 == 0), "ccvpe_colsum: s must be 1 or 2 (even H, W)");
  CCVPE_REQUIRE(dtype == CCVPE_F32 || dtype == CCVPE_BF16, "ccvpe_colsum: bad dtype");
  if (C > 512) {   // wide maps (1024-channel transposed convs, 1280- / 2048-channel cell descriptors): 512 columns per pass
    const int esz = dtype == CCVPE_F32 ? 4 : 2;
    const int buckets = s * s;
    float* tmp = workspace + 4LL * sm_count() * buckets * 512 + 64;    // behind the partials of one 512-column pass
    for (int c0 = 0; c0 < C; c0 += 512) {
      const int cc = C - c0 < 512 ? C - c0 : 512;
      const int rc = ccvpe_colsum(static_cast<const uint8_t*>(x) + (int64_t)c0 * esz, dtype, B, H, W, cc, ld, w, s,
                                  buckets == 1 ? out + c0 : tmp, workspace, stream);
      if (rc != CCVPE_OK) return rc;
      if (buckets > 1) {
        const cudaError_t e = cudaMemcpy2DAsync(out + c0, (size_t)C * 4, tmp, (size_t)cc * 4, (size_t)cc * 4, buckets,
                                                cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
        if (e != cudaSuccess) return fail(CCVPE_ERR_CUDA, "ccvpe_colsum: cudaMemcpy2DAsync: %s", cudaGetErrorString(e));
      }
    }
    return CCVPE_OK;
  }
  const int64_t n_pix = (int64_t)B * H * W;
  CCVPE_REQUIRE(n_pix < (1LL << 31), "ccvpe_colsum: too many pixels");
  const int lanes = CS_THREADS / (C / 4);
  int64_t blocks = (n_pix + 4 * lanes - 1) / (4 * lanes);     // >= 4 pixels per lane, up to 4 blocks per SM
  if (blocks > 4LL * sm_count()) blocks = 4LL * sm_count();
  if (blocks < 1) blocks = 1;
  int64_t ppb = (n_pix + blocks - 1) / blocks;
  ppb = (ppb + lanes - 1) / lanes * lanes;
  blocks = (n_pix + ppb - 1) / ppb;
  const size_t sm = (size_t)lanes * s * s * C * sizeof(float);
  CCVPE_REQUIRE(sm <= 48 * 1024, "ccvpe_colsum: C too large for the block reduction");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CCVPE_F32)
    colsum_partial_kernel<float><<<(int)blocks, CS_THREADS, sm, st>>>((const float*)x, n_pix, H, W, C, ld, w, s, (int)ppb, workspace);
  else
    colsum_partial_kernel<__nv_bfloat16><<<(int)blocks, CS_THREADS, sm, st>>>((const __nv_bfloat16*)x, n_pix, H, W, C, ld, w, s,
                                                                              (int)ppb, workspace);
  CCVPE_LAUNCH_CHECK("colsum_partial_kernel");
  const int n_out = s * s * C;
  colsum_final_kernel<<<(n_out * 32 + 255) / 256, 256, 0, st>>>(workspace, out, n_out, (int)blocks);
  CCVPE_LAUNCH_CHECK("colsum_final_kernel");
  return CCVPE_OK;
}

// ====================================================================================================================
// Pointwise helpers
// ====================================================================================================================
namespace ccvpe {

// dh[i] = h[i] > 0 ? dh[i] : 0      (ReLU backward, in place; 4 elements per thread)
template <typename T>
__global__ void relu_bwd_kernel(T* __restrict__ dh, const T* __restrict__ h, int64_t n4) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g = load4(dh + i * 4);
    const float4 a = load4(h + i * 4);
    g.x = a.x > 0.f ? g.x : 0.f;
    g.y = a.y > 0.f ? g.y : 0.f;
    g.z = a.z > 0.f ? g.z : 0.f;
    g.w = a.w > 0.f ? g.w : 0.f;
    store4(dh + i * 4, g);
  }
}

// planar fp32 [B, N, HW] -> channels-last [B, HW, ld] (channels >= N zero filled)
template <typename T>
__global__ void planar_to_cl_kernel(const float* __restrict__ src, T* __restrict__ dst, int N, int64_t HW, int ld,
                                    int64_t total_pix) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total_pix; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = p / HW, r = p - b * HW;
    for (int c = 0; c < ld; ++c)
      dst[p * ld + c] = from_float<T>(c < N ? src[(b * N + c) * HW + r] : 0.f);
  }
}

// channels-last (dtype) [B, HW, ld] (first N channels) -> planar fp32 [B, N, HW]
template <typename T>
__global__ void cl_to_planar_kernel(const T* __restrict__ src, float* __restrict__ dst, int N, int64_t HW, int ld,
                                    int64_t total_pix) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total_pix; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = p / HW, r = p - b * HW;
    for (int c = 0; c < N; ++c) dst[(b * N + c) * HW + r] = to_float<T>(src[p * ld + c]);
  }
}

// Backward of F.normalize(v, p=2, dim=1, eps=1e-12) on the 2-channel orientation field (reference models.py:341):
//   u = v / max(|v|, eps);   dv = (du - u (u . du)) / |v|         (|v| < eps: dv = du / eps)
// v: channels-last [B, HW, ldv] (first two channels), du: planar fp32 [B, 2, HW]; dv: channels-last (dtype) [B, HW, ldo],
// channels >= 2 zero filled.
template <typename TV, typename TO>
__global__ void ori_normalize_bwd_kernel(const TV* __restrict__ v, int ldv, const float* __restrict__ du,
                                         TO* __restrict__ dv, int ldo, int64_t HW, int64_t total_pix) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total_pix; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = p / HW, r = p - b * HW;
    const float x = to_float<TV>(v[p * ldv]), y = to_float<TV>(v[p * ldv + 1]);
    const float gx = du[(b * 2) * HW + r], gy = du[(b * 2 + 1) * HW + r];
    const float nrm = sqrtf(x * x + y * y);
    float ox, oy;
    if (nrm > 1e-12f) {
      const float inv = 1.f / nrm;
      const float ux = x * inv, uy = y * inv;
      const float dot = ux * gx + uy * gy;
      ox = (gx - ux * dot) * inv;
      oy = (gy - uy * dot) * inv;
    } else {
      ox = gx * 1e12f;
      oy = gy * 1e12f;
    }
    dv[p * ldo] = from_float<TO>(ox);
    dv[p * ldo + 1] = from_float<TO>(oy);
    for (int c = 2; c < ldo; ++c) dv[p * ldo + c] = from_float<TO>(0.f);
  }
}

// y[m, :] = x[m, :] * scale[m]      (the F.normalize'd map as an explicit tensor: the G operand of the tensor-core weight
// gradient of the transposed convs; 4 elements per thread)
template <typename T>
__global__ void scale_rows_kernel(const T* __restrict__ x, const float* __restrict__ scale, T* __restrict__ y, int C4,
                                  int64_t n4) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = load4(x + i * 4);
    const float s = __ldg(scale + i / C4);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    store4(y + i * 4, v);
  }
}

inline int ew_blocks(int64_t n) {
  int64_t b = (n + 255) / 256;
  if (b > 16LL * sm_count()) b = 16LL * sm_count();
  return (int)(b < 1 ? 1 : b);
}

}  // namespace ccvpe

extern "C" int ccvpe_relu_bwd(void* dh, const void* h, int dtype, int64_t n, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(dh && h && n > 0 && n % 4 == 0 && aligned16(dh) && aligned16(h), "ccvpe_relu_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CCVPE_F32) relu_bwd_kernel<float><<<ew_blocks(n / 4), 256, 0, st>>>((float*)dh, (const float*)h, n / 4);
  else if (dtype == CCVPE_BF16)
    relu_bwd_kernel<__nv_bfloat16><<<ew_blocks(n / 4), 256, 0, st>>>((__nv_bfloat16*)dh, (const __nv_bfloat16*)h, n / 4);
  else return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_relu_bwd: bad dtype");
  CCVPE_LAUNCH_CHECK("relu_bwd_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_scale_rows(const void* x, int dtype, const float* scale, void* y, int64_t M, int C, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && scale && y && M > 0 && C > 0 && C % 4 == 0 && aligned16(x) && aligned16(y), "ccvpe_scale_rows: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n4 = M * C / 4;
  if (dtype == CCVPE_F32) scale_rows_kernel<float><<<ew_blocks(n4), 256, 0, st>>>((const float*)x, scale, (float*)y, C / 4, n4);
  else if (dtype == CCVPE_BF16)
    scale_rows_kernel<__nv_bfloat16><<<ew_blocks(n4), 256, 0, st>>>((const __nv_bfloat16*)x, scale, (__nv_bfloat16*)y, C / 4, n4);
  else return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_scale_rows: bad dtype");
  CCVPE_LAUNCH_CHECK("scale_rows_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_planar_to_cl(const float* src, void* dst, int dtype, int B, int N, int64_t HW, int ld, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(src && dst && B > 0 && N > 0 && HW > 0 && ld >= N, "ccvpe_planar_to_cl: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tp = (int64_t)B * HW;
  if (dtype == CCVPE_F32) planar_to_cl_kernel<float><<<ew_blocks(tp), 256, 0, st>>>(src, (float*)dst, N, HW, ld, tp);
  else if (dtype == CCVPE_BF16)
    planar_to_cl_kernel<__nv_bfloat16><<<ew_blocks(tp), 256, 0, st>>>(src, (__nv_bfloat16*)dst, N, HW, ld, tp);
  else return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_planar_to_cl: bad dtype");
  CCVPE_LAUNCH_CHECK("planar_to_cl_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_cl_to_planar(const void* src, int dtype, float* dst, int B, int N, int64_t HW, int ld, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(src && dst && B > 0 && N > 0 && HW > 0 && ld >= N, "ccvpe_cl_to_planar: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tp = (int64_t)B * HW;
  if (dtype == CCVPE_F32) cl_to_planar_kernel<float><<<ew_blocks(tp), 256, 0, st>>>((const float*)src, dst, N, HW, ld, tp);
  else if (dtype == CCVPE_BF16)
    cl_to_planar_kernel<__nv_bfloat16><<<ew_blocks(tp), 256, 0, st>>>((const __nv_bfloat16*)src, dst, N, HW, ld, tp);
  else return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_cl_to_planar: bad dtype");
  CCVPE_LAUNCH_CHECK("cl_to_planar_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_ori_normalize_bwd(const void* v, int v_dtype, int ldv, const float* d_ori, void* dv, int dv_dtype,
                                       int ldo, int B, int64_t HW, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(v && d_ori && dv && B > 0 && HW > 0 && ldv >= 2 && ldo >= 2, "ccvpe_ori_normalize_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t tp = (int64_t)B * HW;
  const int blocks = ew_blocks(tp);
#define CCVPE_ONB(TV, TO) ori_normalize_bwd_kernel<TV, TO><<<blocks, 256, 0, st>>>((const TV*)v, ldv, d_ori, (TO*)dv, ldo, HW, tp)
  if (v_dtype == CCVPE_F32 && dv_dtype == CCVPE_F32) CCVPE_ONB(float, float);
  else if (v_dtype == CCVPE_F32 && dv_dtype == CCVPE_BF16) CCVPE_ONB(float, __nv_bfloat16);
  else if (v_dtype == CCVPE_BF16 && dv_dtype == CCVPE_BF16) CCVPE_ONB(__nv_bfloat16, __nv_bfloat16);
  else if (v_dtype == CCVPE_BF16 && dv_dtype == CCVPE_F32) CCVPE_ONB(__nv_bfloat16, float);
  else return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_ori_normalize_bwd: bad dtype");
#undef CCVPE_ONB
  CCVPE_LAUNCH_CHECK("ori_normalize_bwd_kernel");
  return CCVPE_OK;
}

// ====================================================================================================================
// Backward of one matching level (reference models.py:186-205: the rolled cosine scores, their max over orientations,
// and the F.normalize of the aerial map that is concatenated with the max):
//
//   s_i = <x, G_i> / (n_i * gn),   n_i = ||window_i(x)||,   gn = ||g||,   xhat = x / max(||x||, eps)
//   dS_i  = d_scores_i + [i == argmax over the masked orientations] * d_max
//   dx[c] = inv * (dxhat[c] - xhat[c] * <xhat, dxhat>)  +  sum_i dS_i * ( G_i[c] / (n_i gn) - s_i * M_i[c] * x[c] / n_i^2 )
//   dg[k] = sum_p sum_i dS_i * ( x[p, (k + base_i) % C] / (n_i gn) - s_i * g[k] / gn^2 )
//
// One thread per pixel (128-pixel tiles, like the forward CUDA-core kernel); per 32-channel chunk the tile also accumulates
// T[i][c] = sum_p (dS_i / (n_i gn))[p] * x[p][c], the pixel reduction that dg needs, into a per-tile partial; a finalize
// kernel folds the partials in tile order (deterministic) and applies the circulant re-indexing.
// ====================================================================================================================
namespace ccvpe {

constexpr int MB_TILE = 128;
constexpr int MB_CHUNK = 16;
constexpr int MB_QPR = MB_CHUNK / 4;   // float4 groups per staged row
constexpr int MB_RMAX = 24;

struct MatchBwdArgs {
  const void* x; int HW, C, L, n_rolls; uint32_t max_mask;
  const float* G; const float* Mw; const float* gnorm;       // [B, R, C], [R, C] (NULL when L == C), [B]
  const float* scores;                                       // saved forward scores fp32 [B, R, HW]
  const float* d_scores;                                     // fp32 [B, R, HW] or NULL
  const void* d_max; int ld_dmax;                            // (dtype) [B*HW, ld_dmax] column 0, or NULL
  const void* d_xhat; int ld_dxhat;                          // (dtype) [B*HW, ld_dxhat] first C columns, or NULL
  const void* d_xhat2; int ld_dxhat2;                        // second contribution to d xhat (bottleneck level), or NULL
  const void* d_scores_cl; int ld_dscl;                      // (dtype) [B*HW, ld] columns 0..R-1: channels-last part of dS
  void* dx;                                                  // (dtype) [B, HW, C]
  float* t_part;                                             // [B, tiles, R, C] partial T
  float* c_part;                                             // [B, tiles] partial sum_p sum_i dS_i s_i
  int tiles;
  int csplits, chunks_per_split;                             // pass B (dx, T) is split over channel ranges (blockIdx.z)
};

template <typename T, bool WINDOWED>
__global__ void __launch_bounds__(MB_TILE) match_level_bwd_kernel(const MatchBwdArgs a) {
  __shared__ float xs[MB_TILE][MB_CHUNK + 1];
  __shared__ float ds[MB_TILE][MB_CHUNK + 1];          // d_xhat chunk, then the dx chunk on its way out
  __shared__ __align__(16) float Gs[MB_RMAX][MB_CHUNK];
  __shared__ __align__(16) float Ms[WINDOWED ? MB_RMAX : 1][MB_CHUNK];
  __shared__ float coef_s[MB_RMAX][MB_TILE + 1];       // dS_i / (n_i gn) per pixel

  const int b = blockIdx.y, tile = blockIdx.x;
  const int p0 = tile * MB_TILE;
  const int t = threadIdx.x;
  const int rows = min(MB_TILE, a.HW - p0);
  const int C = a.C, R = a.n_rolls;
  const T* xt = static_cast<const T*>(a.x) + ((int64_t)b * a.HW + p0) * C;
  const T* dxh = a.d_xhat ? static_cast<const T*>(a.d_xhat) + ((int64_t)b * a.HW + p0) * a.ld_dxhat : nullptr;
  const T* dxh2 = a.d_xhat2 ? static_cast<const T*>(a.d_xhat2) + ((int64_t)b * a.HW + p0) * a.ld_dxhat2 : nullptr;
  const float* Gb = a.G + (int64_t)b * R * C;

  auto stage = [&](int c0, bool with_dxhat) {
#pragma unroll
    for (int j = 0; j < (MB_TILE * MB_CHUNK / 4) / MB_TILE; ++j) {
      const int v = t + j * MB_TILE;
      const int row = v / MB_QPR, q = (v % MB_QPR) * 4;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f), dval = val;
      if (row < rows && c0 + q < C) {
        val = load4(xt + (int64_t)row * C + c0 + q);
        if (with_dxhat && dxh) dval = load4(dxh + (int64_t)row * a.ld_dxhat + c0 + q);
        if (with_dxhat && dxh2) {
          const float4 e = load4(dxh2 + (int64_t)row * a.ld_dxhat2 + c0 + q);
          dval.x += e.x; dval.y += e.y; dval.z += e.z; dval.w += e.w;
        }
      }
      xs[row][q] = val.x; xs[row][q + 1] = val.y; xs[row][q + 2] = val.z; xs[row][q + 3] = val.w;
      if (with_dxhat) { ds[row][q] = dval.x; ds[row][q + 1] = dval.y; ds[row][q + 2] = dval.z; ds[row][q + 3] = dval.w; }
    }
    for (int v = t; v < MB_RMAX * MB_QPR; v += MB_TILE) {
      const int i = v / MB_QPR, q = (v % MB_QPR) * 4;
      float4 gv = make_float4(0.f, 0.f, 0.f, 0.f), mv = gv;
      if (i < R && c0 + q < C) {
        gv = *reinterpret_cast<const float4*>(Gb + (int64_t)i * C + c0 + q);
        if (WINDOWED) mv = *reinterpret_cast<const float4*>(a.Mw + (int64_t)i * C + c0 + q);
      }
      *reinterpret_cast<float4*>(&Gs[i][q]) = gv;
      if (WINDOWED) *reinterpret_cast<float4*>(&Ms[i][q]) = mv;
    }
  };

  // ---- pass A: ||x||^2, window norms, <x, d_xhat> ----
  float sq = 0.f, dot = 0.f;
  float wsq[WINDOWED ? MB_RMAX : 1];
#pragma unroll
  for (int i = 0; i < (WINDOWED ? MB_RMAX : 1); ++i) wsq[i] = 0.f;
  for (int c0 = 0; c0 < C; c0 += MB_CHUNK) {
    stage(c0, true);
    __syncthreads();
#pragma unroll 4
    for (int cc = 0; cc < MB_CHUNK; ++cc) {
      const float xv = xs[t][cc];
      const float x2 = xv * xv;
      sq += x2;
      dot = fmaf(xv, ds[t][cc], dot);
      if (WINDOWED) {
#pragma unroll
        for (int i = 0; i < MB_RMAX; ++i) wsq[i] = fmaf(x2, Ms[i][cc], wsq[i]);
      }
    }
    __syncthreads();
  }
  // ---- per-pixel coefficients ----
  const float gn = a.gnorm[b];
  const float nrm = sqrtf(sq);
  const bool tiny = !(nrm > 1e-12f);
  const float inv = tiny ? 1e12f : 1.f / nrm;
  const float k_self = tiny ? 0.f : inv * inv * inv * dot;       // coefficient of x[c] from the normalise backward
  float beta_all = 0.f;                                           // sum_i dS_i s_i / n_i^2     (full-circle: n_i = ||x||)
  float beta[WINDOWED ? MB_RMAX : 1];
  float cpart = 0.f;                                              // sum_i dS_i s_i
  {
    const int64_t pix = (int64_t)b * a.HW + p0 + t;
    float dmax = 0.f;
    int arg = -1;
    if (t < rows && a.d_max) {
      dmax = to_float<T>(static_cast<const T*>(a.d_max)[pix * a.ld_dmax]);
      float best = -INFINITY;
      for (int i = 0; i < R; ++i) {
        if (!((a.max_mask >> i) & 1u)) continue;
        const float s = a.scores[((int64_t)b * R + i) * a.HW + p0 + t];
        if (s > best || (arg < 0)) {   // first maximum wins (torch.max returns the first index of the maximum)
          if (arg < 0 || s > best) { best = s; arg = i; }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < MB_RMAX; ++i) {
      float co = 0.f, be = 0.f;
      if (i < R && t < rows) {
        const int64_t si = ((int64_t)b * R + i) * a.HW + p0 + t;
        float dS = a.d_scores ? a.d_scores[si] : 0.f;
        if (a.d_scores_cl) dS += to_float<T>(static_cast<const T*>(a.d_scores_cl)[pix * a.ld_dscl + i]);
        if (i == arg) dS += dmax;
        const float s = a.scores[si];
        const float n2 = WINDOWED ? wsq[i] : sq;
        const float n = sqrtf(n2);
        co = dS / (n * gn);
        be = dS * s / n2;
        cpart += dS * s;
        if (dS == 0.f) { co = 0.f; be = 0.f; }        // (zero windows: 0 * inf must not poison the gradient)
      }
      coef_s[i][t] = co;
      if (WINDOWED) beta[i] = be; else beta_all += be;
    }
  }
  // deterministic block reduction of cpart (tile order is fixed; lanes are folded in a fixed tree)
  {
    __shared__ float red[MB_TILE / 32];
    float v = warp_sum(cpart);
    if ((t & 31) == 0) red[t >> 5] = v;
    __syncthreads();
    if (t == 0 && blockIdx.z == 0) a.c_part[(int64_t)b * a.tiles + tile] = (red[0] + red[1]) + (red[2] + red[3]);
  }
  __syncthreads();
  // ---- pass B: dx and the partial T ----
  T* dxo = static_cast<T*>(a.dx) + ((int64_t)b * a.HW + p0) * C;
  float* tp = a.t_part + ((int64_t)b * a.tiles + tile) * R * C;
  // small maps have few pixel tiles: the channel axis of this pass is split over blockIdx.z (pass A above is cheap and is
  // simply repeated by every split)
  const int cb_begin = blockIdx.z * a.chunks_per_split * MB_CHUNK;
  const int cb_end = min(C, cb_begin + a.chunks_per_split * MB_CHUNK);
  for (int c0 = cb_begin; c0 < cb_end; c0 += MB_CHUNK) {
    stage(c0, true);
    __syncthreads();
    // (1) T[i][c0 + cc] partial: R x 32 outputs, each a 128-term dot product over the tile's pixels
    for (int o = t; o < R * MB_CHUNK; o += MB_TILE) {
      const int i = o / MB_CHUNK, cc = o - i * MB_CHUNK;
      float s = 0.f;
#pragma unroll 8
      for (int p = 0; p < MB_TILE; ++p) s = fmaf(coef_s[i][p], xs[p][cc], s);
      if (c0 + cc < C) tp[(int64_t)i * C + c0 + cc] = s;
    }
    // (2) dx of this thread's pixel
    float outv[MB_CHUNK];
#pragma unroll
    for (int cc = 0; cc < MB_CHUNK; ++cc) {
      const float xv = xs[t][cc];
      float v = inv * ds[t][cc] - k_self * xv;
      float gsum = 0.f, msum = WINDOWED ? 0.f : beta_all;
#pragma unroll
      for (int i = 0; i < MB_RMAX; ++i) {
        gsum = fmaf(coef_s[i][t], Gs[i][cc], gsum);
        if (WINDOWED) msum = fmaf(beta[i], Ms[i][cc], msum);
      }
      outv[cc] = v + gsum - msum * xv;
    }
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < MB_CHUNK; ++cc) ds[t][cc] = outv[cc];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < (MB_TILE * MB_CHUNK / 4) / MB_TILE; ++j) {
      const int v = t + j * MB_TILE;
      const int row = v / MB_QPR, q = (v % MB_QPR) * 4;
      if (row < rows && c0 + q < C)
        store4(dxo + (int64_t)row * C + c0 + q, make_float4(ds[row][q], ds[row][q + 1], ds[row][q + 2], ds[row][q + 3]));
    }
    __syncthreads();
  }
}

struct RollShifts {
  int s[32];
};

// T_sum[b][e] = sum_tiles t_part[b][tile][e] (e over R*C), tiles in order: one thread per (b, e), coalesced over e
__global__ void match_bwd_reduce_tiles_kernel(const float* __restrict__ t_part, int tiles, int RC, float* __restrict__ t_sum) {
  const int b = blockIdx.y;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < RC; e += gridDim.x * blockDim.x) {
    const float* src = t_part + (int64_t)b * tiles * RC + e;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int tl = 0;
    for (; tl + 4 <= tiles; tl += 4) {       // four independent chains (fixed association: deterministic)
      s0 += src[(int64_t)tl * RC];
      s1 += src[(int64_t)(tl + 1) * RC];
      s2 += src[(int64_t)(tl + 2) * RC];
      s3 += src[(int64_t)(tl + 3) * RC];
    }
    for (; tl < tiles; ++tl) s0 += src[(int64_t)tl * RC];
    t_sum[(int64_t)b * RC + e] = (s0 + s1) + (s2 + s3);
  }
}

// dg[b, k] = sum_i T_sum[b, i, (k + base_i) % C]  -  g[b, k] / gn^2 * sum_tiles c_part[b, tile]
// (T already carries the 1 / (n_i gn) of the per-pixel coefficients)
__global__ void match_bwd_finalize_kernel(const float* __restrict__ t_sum, const float* __restrict__ c_part, int tiles,
                                          int R, int C, int L, int offset, RollShifts sh, const float* __restrict__ g,
                                          const float* __restrict__ gnorm, float* __restrict__ dg) {
  const int b = blockIdx.y;
  const float gn = gnorm[b];
  float csum = 0.f;
  for (int tl = 0; tl < tiles; ++tl) csum += c_part[(int64_t)b * tiles + tl];
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < L; k += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < R; ++i) {
      const int base = ((offset + sh.s[i]) % C + C) % C;
      int c = k + base;
      if (c >= C) c -= C;
      s += t_sum[((int64_t)b * R + i) * C + c];
    }
    dg[(int64_t)b * L + k] = s - g[(int64_t)b * L + k] * csum / (gn * gn);
  }
}

// defined in match.cu
struct RollTableFwd;
int build_rolled_descriptor_f32(const float* g, int B, int L, int C, int offset, const int32_t* shifts_host, int n_rolls,
                                float* G, float* M, float* gnorm, cudaStream_t st);

}  // namespace ccvpe

extern "C" int64_t ccvpe_match_bwd_scratch_elems(int B, int HW, int C, int n_rolls) {
  auto up = [](int64_t v) { return (v + 63) / 64 * 64; };
  const int64_t tiles = (HW + 127) / 128;
  return up((int64_t)B * n_rolls * C) + up((int64_t)n_rolls * C) + up(B) + up((int64_t)B * tiles * n_rolls * C) +
         up((int64_t)B * tiles) + up((int64_t)B * n_rolls * C) + 256;
}

extern "C" int ccvpe_match_level_bwd(const void* x, int dtype, int B, int HW, int C, const float* g, int L, int offset,
                                     const int32_t* shifts_host, int n_rolls, uint32_t max_mask, const float* scores,
                                     const float* d_scores, const void* d_scores_cl, int ld_dscl, const void* d_max,
                                     int ld_dmax, const void* d_xhat, int ld_dxhat, const void* d_xhat2, int ld_dxhat2,
                                     void* dx, float* dg, float* scratch, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && g && shifts_host && scores && dx && dg && scratch, "ccvpe_match_level_bwd: null pointer");
  CCVPE_REQUIRE(B > 0 && HW > 0 && C > 0 && C % 8 == 0 && L > 0 && L <= C, "ccvpe_match_level_bwd: bad shape");
  CCVPE_REQUIRE(n_rolls > 0 && n_rolls <= MB_RMAX, "ccvpe_match_level_bwd: n_rolls=%d out of range", n_rolls);
  CCVPE_REQUIRE(dtype == CCVPE_F32 || dtype == CCVPE_BF16, "ccvpe_match_level_bwd: bad dtype");
  CCVPE_REQUIRE(!d_xhat || (ld_dxhat >= C && ld_dxhat % 4 == 0), "ccvpe_match_level_bwd: bad d_xhat stride");
  CCVPE_REQUIRE(!d_xhat2 || (d_xhat && ld_dxhat2 >= C && ld_dxhat2 % 4 == 0), "ccvpe_match_level_bwd: bad d_xhat2");
  CCVPE_REQUIRE(!d_scores_cl || ld_dscl >= n_rolls, "ccvpe_match_level_bwd: bad d_scores_cl stride");
  CCVPE_REQUIRE(!d_max || ld_dmax >= 1, "ccvpe_match_level_bwd: bad d_max stride");
  cudaStream_t st = (cudaStream_t)stream;
  auto up = [](int64_t v) { return (v + 63) / 64 * 64; };
  const int tiles = (HW + MB_TILE - 1) / MB_TILE;
  float* G = scratch;
  float* Mw = G + up((int64_t)B * n_rolls * C);
  float* gnorm = Mw + up((int64_t)n_rolls * C);
  float* t_part = gnorm + up(B);
  float* c_part = t_part + up((int64_t)B * tiles * n_rolls * C);
  float* t_sum = c_part + up((int64_t)B * tiles);
  const bool windowed = L < C;
  int rc = build_rolled_descriptor_f32(g, B, L, C, offset, shifts_host, n_rolls, G, windowed ? Mw : nullptr, gnorm, st);
  if (rc != CCVPE_OK) return rc;
  MatchBwdArgs a;
  a.x = x; a.HW = HW; a.C = C; a.L = L; a.n_rolls = n_rolls; a.max_mask = max_mask;
  a.G = G; a.Mw = windowed ? Mw : nullptr; a.gnorm = gnorm;
  a.scores = scores; a.d_scores = d_scores;
  a.d_max = d_max; a.ld_dmax = ld_dmax; a.d_xhat = d_xhat; a.ld_dxhat = ld_dxhat;
  a.d_xhat2 = d_xhat2; a.ld_dxhat2 = ld_dxhat2; a.d_scores_cl = d_scores_cl; a.ld_dscl = ld_dscl;
  a.dx = dx; a.t_part = t_part; a.c_part = c_part; a.tiles = tiles;
  const int chunks = (C + MB_CHUNK - 1) / MB_CHUNK;
  int csplits = (2 * sm_count() + tiles * B - 1) / (tiles * B);
  if (csplits > chunks) csplits = chunks;
  if (csplits < 1) csplits = 1;
  a.chunks_per_split = (chunks + csplits - 1) / csplits;
  a.csplits = (chunks + a.chunks_per_split - 1) / a.chunks_per_split;
  const dim3 grid(tiles, B, a.csplits);
#define CCVPE_MB(TT, WW) match_level_bwd_kernel<TT, WW><<<grid, MB_TILE, 0, st>>>(a)
  if (dtype == CCVPE_F32) { if (windowed) CCVPE_MB(float, true); else CCVPE_MB(float, false); }
  else { if (windowed) CCVPE_MB(__nv_bfloat16, true); else CCVPE_MB(__nv_bfloat16, false); }
#undef CCVPE_MB
  CCVPE_LAUNCH_CHECK("match_level_bwd_kernel");
  RollShifts sh;
  for (int i = 0; i < 32; ++i) sh.s[i] = i < n_rolls ? shifts_host[i] : 0;
  const int RC = n_rolls * C;
  match_bwd_reduce_tiles_kernel<<<dim3((RC + 255) / 256, B), 256, 0, st>>>(t_part, tiles, RC, t_sum);
  CCVPE_LAUNCH_CHECK("match_bwd_reduce_tiles_kernel");
  match_bwd_finalize_kernel<<<dim3((L + 127) / 128, B), 128, 0, st>>>(t_sum, c_part, tiles, n_rolls, C, L, offset, sh, g,
                                                                      gnorm, dg);
  CCVPE_LAUNCH_CHECK("match_bwd_finalize_kernel");
  return CCVPE_OK;
}

// ====================================================================================================================
// Training losses, forward + gradient in one call (reference losses.py:4-29).  Each is: a partial kernel over chunks of the
// flattened row (per-sample statistics to the workspace), a one-block finalize (fixed order), and a gradient pass.
// stats layout (fp32, in `workspace`): see the kernels.  `loss` receives the scalar; gradients are d loss / d input.
// ====================================================================================================================
namespace ccvpe {

constexpr int LS_THREADS = 256;

__device__ __forceinline__ float block_sum_256(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  if (threadIdx.x == 0) {
    for (int i = 0; i < LS_THREADS / 32; ++i) r += red[i];
  }
  __syncthreads();
  return r;   // valid in thread 0
}

// How the InfoNCE kernels fetch label j of row b (j = flat index into the row of n = R * hw labels).
//   DenseLabels:  lab [B, n], the max-pooled orientation-binned map as stored.
//   BinnedLabels: the rank-1 form of the same map, pooled [B, hw] (the pooled location map) times w [B, R] (the pair's bin
//                 weights).  __fmul_rn is the correctly rounded product that the dense map's `gt * w` stores (max-pooling
//                 commutes with it: rounding is monotone and w >= 0), and it keeps nvcc from contracting it into the
//                 `w += l` / fmaf that follow, so both give the same label bits.
struct DenseLabels {
  const float* lab;
  int64_t n;
  __device__ __forceinline__ float operator()(int b, int64_t j) const { return lab[b * n + j]; }
};
struct BinnedLabels {
  const float* pooled;
  const float* w;
  int R;
  uint32_t hw;                                     // R * hw < 2^31 (checked by the launcher)
  __device__ __forceinline__ float operator()(int b, int64_t j) const {
    const uint32_t r = (uint32_t)j / hw, p = (uint32_t)j - r * hw;
    return __fmul_rn(pooled[(int64_t)b * hw + p], w[b * R + r]);
  }
};

// infoNCE (losses.py:4-20): per (row b, chunk): sum exp(s / tau), sum w, sum w * s / tau       (w = label if label > 1e-2)
template <typename Labels>
__global__ void __launch_bounds__(LS_THREADS)
infonce_partial_kernel(const float* __restrict__ s, const Labels lab, int64_t n, int chunks, float inv_tau,
                       float* __restrict__ part) {
  __shared__ float red[LS_THREADS / 32];
  const int b = blockIdx.y, ch = blockIdx.x;
  const int64_t per = (n + chunks - 1) / chunks;
  const int64_t lo = ch * per, hi = min(n, lo + per);
  float e = 0.f, w = 0.f, ws = 0.f;
  for (int64_t j = lo + threadIdx.x; j < hi; j += LS_THREADS) {
    const float v = s[b * n + j] * inv_tau;
    const float l = lab(b, j);
    e += __expf(v);
    if (l > 1e-2f) {
      w += l;
      ws = fmaf(l, v, ws);
    }
  }
  const float e_t = block_sum_256(e, red), w_t = block_sum_256(w, red), ws_t = block_sum_256(ws, red);
  if (threadIdx.x == 0) {
    float* o = part + ((int64_t)b * chunks + ch) * 3;
    o[0] = e_t; o[1] = w_t; o[2] = ws_t;
  }
}

// stats[b*2] = sum exp, stats[b*2+1] = sum w;  stats[2B] = W = total weight;  loss
__global__ void infonce_finalize_kernel(const float* __restrict__ part, int B, int chunks, float* __restrict__ stats,
                                        float* __restrict__ loss) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float W = 0.f, num = 0.f;
  for (int b = 0; b < B; ++b) {
    float e = 0.f, w = 0.f, ws = 0.f;
    for (int c = 0; c < chunks; ++c) {
      const float* o = part + ((int64_t)b * chunks + c) * 3;
      e += o[0]; w += o[1]; ws += o[2];
    }
    stats[b * 2] = e;
    stats[b * 2 + 1] = w;
    W += w;
    num += ws - w * logf(e);
  }
  stats[2 * B] = W;
  *loss = -num / W;
}

// d loss / d s[b, j] = -(1 / W) * ( w_j / tau - (sum_b w) * exp(s_j / tau) / (tau * sum_b exp) )
template <typename Labels>
__global__ void infonce_grad_kernel(const float* __restrict__ s, const Labels lab, int64_t n, int B,
                                    float inv_tau, const float* __restrict__ stats, float* __restrict__ ds) {
  const float W = stats[2 * B];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)B * n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / n);
    const float v = s[i] * inv_tau;
    const float l = lab(b, i - b * n);
    const float w = l > 1e-2f ? l : 0.f;
    ds[i] = -(w - stats[b * 2 + 1] * __expf(v) / stats[b * 2]) * inv_tau / W;
  }
}

// cross entropy (losses.py:23-24): -sum(labels * log_softmax(logits)) / B.  Partials per (b, chunk): max, sum exp(l - max),
// sum labels, sum labels * logits
__global__ void __launch_bounds__(LS_THREADS)
ce_partial_kernel(const float* __restrict__ lg, const float* __restrict__ lab, int64_t n, int chunks, float* __restrict__ part) {
  __shared__ float red[LS_THREADS / 32];
  __shared__ float s_max;
  const int b = blockIdx.y, ch = blockIdx.x;
  const int64_t per = (n + chunks - 1) / chunks;
  const int64_t lo = ch * per, hi = min(n, lo + per);
  float mx = -INFINITY;
  for (int64_t j = lo + threadIdx.x; j < hi; j += LS_THREADS) mx = fmaxf(mx, lg[b * n + j]);
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < LS_THREADS / 32; ++i) m = fmaxf(m, red[i]);
    s_max = m;
  }
  __syncthreads();
  const float M = s_max;
  float e = 0.f, sl = 0.f, sll = 0.f;
  for (int64_t j = lo + threadIdx.x; j < hi; j += LS_THREADS) {
    const float v = lg[b * n + j], l = lab[b * n + j];
    e += __expf(v - M);
    sl += l;
    sll = fmaf(l, v, sll);
  }
  const float e_t = block_sum_256(e, red), sl_t = block_sum_256(sl, red), sll_t = block_sum_256(sll, red);
  if (threadIdx.x == 0) {
    float* o = part + ((int64_t)b * chunks + ch) * 4;
    o[0] = M; o[1] = e_t; o[2] = sl_t; o[3] = sll_t;
  }
}

// stats[b*3] = max, [b*3+1] = sum exp(l - max), [b*3+2] = sum labels
__global__ void ce_finalize_kernel(const float* __restrict__ part, int B, int chunks, float* __restrict__ stats,
                                   float* __restrict__ loss) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float total = 0.f;
  for (int b = 0; b < B; ++b) {
    float M = -INFINITY;
    for (int c = 0; c < chunks; ++c) M = fmaxf(M, part[((int64_t)b * chunks + c) * 4]);
    float e = 0.f, sl = 0.f, sll = 0.f;
    for (int c = 0; c < chunks; ++c) {
      const float* o = part + ((int64_t)b * chunks + c) * 4;
      e += o[1] * __expf(o[0] - M);
      sl += o[2];
      sll += o[3];
    }
    stats[b * 3] = M; stats[b * 3 + 1] = e; stats[b * 3 + 2] = sl;
    total += sll - sl * (M + logf(e));          // sum labels * (logit - logsumexp)
  }
  *loss = -total / (float)B;
}

// d loss / d logit = (softmax * sum(labels) - labels) / B
__global__ void ce_grad_kernel(const float* __restrict__ lg, const float* __restrict__ lab, int64_t n, int B,
                               const float* __restrict__ stats, float* __restrict__ dl) {
  const float invB = 1.f / (float)B;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)B * n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / n);
    const float p = __expf(lg[i] - stats[b * 3]) / stats[b * 3 + 1];
    dl[i] = (p * stats[b * 3 + 2] - lab[i]) * invB;
  }
}

// How ori_loss_kernel fetches the target (c = 0: cos, 1: sin) of pair b at pixel r.
//   DenseOrientation: gt_ori planar [B, 2, HW], the orientation field as stored.
//   ConstOrientation: v [B, 2], one unit vector per pair (the field is constant over the map).
struct DenseOrientation {
  const float* gt_ori;
  int64_t HW;
  __device__ __forceinline__ float operator()(int64_t b, int c, int64_t r) const { return gt_ori[(b * 2 + c) * HW + r]; }
};
struct ConstOrientation {
  const float* v;
  __device__ __forceinline__ float operator()(int64_t b, int c, int64_t) const { return v[b * 2 + c]; }
};

// orientation loss (losses.py:28-29): sum_p gt[p] * ((go0 - o0)^2 + (go1 - o1)^2) / B; partial per block
template <typename Target>
__global__ void __launch_bounds__(LS_THREADS)
ori_loss_kernel(const float* __restrict__ ori, const Target gt_ori, const float* __restrict__ gt, int64_t HW,
                int B, float* __restrict__ part, float* __restrict__ d_ori) {
  __shared__ float red[LS_THREADS / 32];
  const float invB = 1.f / (float)B;
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)B * HW; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / HW, r = i - b * HW;
    const float w = gt[i];
    const float e0 = gt_ori(b, 0, r) - ori[(b * 2) * HW + r];
    const float e1 = gt_ori(b, 1, r) - ori[(b * 2 + 1) * HW + r];
    acc = fmaf(w, e0 * e0 + e1 * e1, acc);
    d_ori[(b * 2) * HW + r] = -2.f * w * e0 * invB;
    d_ori[(b * 2 + 1) * HW + r] = -2.f * w * e1 * invB;
  }
  const float tot = block_sum_256(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = tot;
}

__global__ void sum_scale_kernel(const float* __restrict__ part, int n, float scale, float* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float s = 0.f;
  for (int i = 0; i < n; ++i) s += part[i];
  *out = s * scale;
}

constexpr int LS_MAX_CHUNKS = 64;
inline int loss_chunks(int B, int64_t n) {
  int c = (2 * sm_count() + B - 1) / B;
  if (c > LS_MAX_CHUNKS) c = LS_MAX_CHUNKS;
  const int64_t maxc = (n + 4095) / 4096;
  if (c > maxc) c = (int)maxc;
  return c < 1 ? 1 : c;
}

}  // namespace ccvpe

extern "C" int64_t ccvpe_loss_workspace_elems(int B) { return (int64_t)B * ccvpe::LS_MAX_CHUNKS * 4 + 4 * B + 2048; }

namespace ccvpe {

template <typename Labels>
static int infonce_launch(const float* scores, const Labels lab, int B, int64_t n, float temperature, float* loss,
                          float* d_scores, float* workspace, cudaStream_t st) {
  const int chunks = loss_chunks(B, n);
  float* part = workspace;
  float* stats = workspace + (int64_t)B * LS_MAX_CHUNKS * 4;
  infonce_partial_kernel<<<dim3(chunks, B), LS_THREADS, 0, st>>>(scores, lab, n, chunks, 1.f / temperature, part);
  CCVPE_LAUNCH_CHECK("infonce_partial_kernel");
  infonce_finalize_kernel<<<1, 32, 0, st>>>(part, B, chunks, stats, loss);
  CCVPE_LAUNCH_CHECK("infonce_finalize_kernel");
  infonce_grad_kernel<<<ew_blocks((int64_t)B * n), 256, 0, st>>>(scores, lab, n, B, 1.f / temperature, stats, d_scores);
  CCVPE_LAUNCH_CHECK("infonce_grad_kernel");
  return CCVPE_OK;
}

template <typename Target>
static int ori_loss_launch(const float* ori, const Target gt_ori, const float* gt, int B, int64_t HW, float* loss,
                           float* d_ori, float* workspace, cudaStream_t st) {
  int blocks = ew_blocks((int64_t)B * HW);
  if (blocks > 1024) blocks = 1024;
  ori_loss_kernel<<<blocks, LS_THREADS, 0, st>>>(ori, gt_ori, gt, HW, B, workspace, d_ori);
  CCVPE_LAUNCH_CHECK("ori_loss_kernel");
  sum_scale_kernel<<<1, 32, 0, st>>>(workspace, blocks, 1.f / (float)B, loss);
  CCVPE_LAUNCH_CHECK("sum_scale_kernel");
  return CCVPE_OK;
}

}  // namespace ccvpe

extern "C" int ccvpe_infonce_loss(const float* scores, const float* labels, int B, int64_t n, float temperature, float* loss,
                                  float* d_scores, float* workspace, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(scores && labels && loss && d_scores && workspace && B > 0 && n > 0 && temperature > 0.f,
                "ccvpe_infonce_loss: bad argument");
  return infonce_launch(scores, DenseLabels{labels, n}, B, n, temperature, loss, d_scores, workspace, (cudaStream_t)stream);
}

extern "C" int ccvpe_infonce_loss_binned(const float* scores, const float* pooled, const float* bin_w, int B, int R,
                                         int64_t HW, float temperature, float* loss, float* d_scores, float* workspace,
                                         void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(scores && pooled && bin_w && loss && d_scores && workspace && B > 0 && R > 0 && HW > 0 &&
                    (int64_t)R * HW <= INT32_MAX && temperature > 0.f,
                "ccvpe_infonce_loss_binned: bad argument (B=%d, R=%d, HW=%lld)", B, R, (long long)HW);
  const int64_t n = (int64_t)R * HW;
  return infonce_launch(scores, BinnedLabels{pooled, bin_w, R, (uint32_t)HW}, B, n, temperature, loss, d_scores, workspace,
                        (cudaStream_t)stream);
}

extern "C" int ccvpe_cross_entropy_loss(const float* logits, const float* labels, int B, int64_t n, float* loss,
                                        float* d_logits, float* workspace, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(logits && labels && loss && d_logits && workspace && B > 0 && n > 0, "ccvpe_cross_entropy_loss: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = loss_chunks(B, n);
  float* part = workspace;
  float* stats = workspace + (int64_t)B * LS_MAX_CHUNKS * 4;
  ce_partial_kernel<<<dim3(chunks, B), LS_THREADS, 0, st>>>(logits, labels, n, chunks, part);
  CCVPE_LAUNCH_CHECK("ce_partial_kernel");
  ce_finalize_kernel<<<1, 32, 0, st>>>(part, B, chunks, stats, loss);
  CCVPE_LAUNCH_CHECK("ce_finalize_kernel");
  ce_grad_kernel<<<ew_blocks((int64_t)B * n), 256, 0, st>>>(logits, labels, n, B, stats, d_logits);
  CCVPE_LAUNCH_CHECK("ce_grad_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_orientation_loss(const float* ori, const float* gt_ori, const float* gt, int B, int64_t HW, float* loss,
                                      float* d_ori, float* workspace, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(ori && gt_ori && gt && loss && d_ori && workspace && B > 0 && HW > 0, "ccvpe_orientation_loss: bad argument");
  return ori_loss_launch(ori, DenseOrientation{gt_ori, HW}, gt, B, HW, loss, d_ori, workspace, (cudaStream_t)stream);
}

extern "C" int ccvpe_orientation_loss_const(const float* ori, const float* ori_vec, const float* gt, int B, int64_t HW,
                                            float* loss, float* d_ori, float* workspace, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(ori && ori_vec && gt && loss && d_ori && workspace && B > 0 && HW > 0,
                "ccvpe_orientation_loss_const: bad argument");
  return ori_loss_launch(ori, ConstOrientation{ori_vec}, gt, B, HW, loss, d_ori, workspace, (cudaStream_t)stream);
}

// ====================================================================================================================
// Label pyramid of the InfoNCE terms (reference train_VIGOR.py:128-133, max_pool2d(gt, k, stride=k) for k = 64 ... 2) in one
// pass: each CTA loads one 64x64 tile of gt [B, H, W] with float4 loads and halves it 2x2 by 2x2 in shared memory, writing
// every level on the way.  Level l (k = 64 >> l) is [B, H/k, W/k] at element offset B * sum_{m<l} (H / k_m) * (W / k_m) of
// `out`.  The max propagates NaN like max_pool2d: any NaN in a window gives NaN.
// ====================================================================================================================
namespace ccvpe {

constexpr int PYR_TILE = 64, PYR_THREADS = 256, PYR_LEVELS = 6;

__device__ __forceinline__ float max_nan(float a, float b) { return (a > b || a != a) ? a : b; }

__host__ __device__ __forceinline__ int64_t pyr_level_offset(int l, int B, int H, int W) {
  int64_t off = 0;
  for (int m = 0; m < l; ++m) off += (int64_t)B * (H >> (PYR_LEVELS - m)) * (W >> (PYR_LEVELS - m));
  return off;
}

__global__ void __launch_bounds__(PYR_THREADS) gt_pyramid_kernel(const float* __restrict__ gt, int H, int W,
                                                                 float* __restrict__ out) {
  __shared__ float4 tile4[PYR_TILE * PYR_TILE / 4];
  __shared__ float halved[PYR_TILE * PYR_TILE / 4];
  float* tile = reinterpret_cast<float*>(tile4);
  const int tx = blockIdx.x, ty = blockIdx.y, b = blockIdx.z, B = gridDim.z;
  const float* src = gt + ((int64_t)b * H + (int64_t)ty * PYR_TILE) * W + (int64_t)tx * PYR_TILE;
#pragma unroll
  for (int i = 0; i < PYR_TILE * PYR_TILE / 4 / PYR_THREADS; ++i) {
    const int q = threadIdx.x + i * PYR_THREADS, row = q / (PYR_TILE / 4), c4 = q % (PYR_TILE / 4);
    tile4[q] = __ldg(reinterpret_cast<const float4*>(src + (int64_t)row * W) + c4);
  }
  __syncthreads();
  // level l = 5 .. 0 (k = 2 .. 64): this tile's n x n map (n = 64 / k) is reduced from the 2n x 2n one, ping-ponging
  // tile <-> halved
  float* cur = tile;
  float* nxt = halved;
  for (int l = PYR_LEVELS - 1; l >= 0; --l) {
    const int n = 1 << l, Hl = H >> (PYR_LEVELS - l), Wl = W >> (PYR_LEVELS - l);
    float* dst = out + pyr_level_offset(l, B, H, W) + ((int64_t)b * Hl + (int64_t)ty * n) * Wl + (int64_t)tx * n;
    for (int q = threadIdx.x; q < n * n; q += PYR_THREADS) {
      const int y = q >> l, x = q & (n - 1);
      const float* c = cur + (2 * y) * (2 * n) + 2 * x;
      const float m = max_nan(max_nan(c[0], c[1]), max_nan(c[2 * n], c[2 * n + 1]));
      nxt[q] = m;
      dst[(int64_t)y * Wl + x] = m;
    }
    __syncthreads();
    float* t = cur;
    cur = nxt;
    nxt = t;
  }
}

}  // namespace ccvpe

extern "C" int ccvpe_gt_pyramid(const float* gt, int B, int H, int W, float* out, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(gt && out && B > 0 && H > 0 && W > 0 && H % PYR_TILE == 0 && W % PYR_TILE == 0 && B <= 65535 &&
                    H / PYR_TILE <= 65535 && ((uintptr_t)gt & 15) == 0,
                "ccvpe_gt_pyramid: bad argument (B=%d, H=%d, W=%d: H and W must be positive multiples of %d, gt 16-byte "
                "aligned)", B, H, W, PYR_TILE);
  gt_pyramid_kernel<<<dim3(W / PYR_TILE, H / PYR_TILE, B), PYR_THREADS, 0, (cudaStream_t)stream>>>(gt, H, W, out);
  CCVPE_LAUNCH_CHECK("gt_pyramid_kernel");
  return CCVPE_OK;
}

// ====================================================================================================================
// Backward of the ground descriptor heads (reference models.py:57-97, 152-157):
//   g_l[b, w*c_l + ch] = sum_h v_l[h] * (sum_k W_l[ch, k] * F[b, k, h, w] + b1_l[ch]) + b2_l
// With dT_l[b, ch, w] = dg_l[b, w*c_l + ch] and P_l[b, k, w] = sum_h v_l[h] F[b, k, h, w] (the forward's height-reduced
// scratch, recomputed here) and U_l[b, k, w] = sum_ch W_l[ch, k] dT_l[b, ch, w]:
//   dF[b, k, h, w] = sum_l v_l[h] U_l[b, k, w]          dW_l[ch, k] = sum_{b, w} dT_l[b, ch, w] P_l[b, k, w]
//   db1_l[ch] = (sum_h v_l[h]) sum_{b, w} dT_l          db2_l = sum dg_l
//   dv_l[h] = sum_{b, k, w} F[b, k, h, w] U_l[b, k, w] + sum_{b, ch, w} dT_l[b, ch, w] b1_l[ch]
// Tiny (64 MFLOP per pair forward): plain kernels, deterministic (no atomics: one thread / block per output).
// ====================================================================================================================
namespace ccvpe {

struct HeadsBwdArgs {
  const void* feat; int dtype; int B, K, H, W; int64_t sb, sk, sh, sw;
  int n_heads;
  const float* w1[6]; const float* b1[6]; const float* w2[6];
  const float* dg[6];
  int c[6];
  float* U;        // [n_heads, B, K, W]
  float* dfeat;    // fp32 [B, K, H, W] contiguous
  float* dw1[6]; float* db1[6]; float* dw2[6]; float* db2[6];
};

template <typename T>
__device__ __forceinline__ float feat_at(const HeadsBwdArgs& a, int b, int k, int h, int w) {
  return to_float<T>(static_cast<const T*>(a.feat)[b * a.sb + k * a.sk + h * a.sh + w * a.sw]);
}

// U_l[b, k, w] and dF[b, k, h, w]: one thread per (b, k, w)
template <typename T>
__global__ void heads_bwd_data_kernel(const HeadsBwdArgs a) {
  const int64_t total = (int64_t)a.B * a.K * a.W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % a.W);
    const int k = (int)((i / a.W) % a.K);
    const int b = (int)(i / ((int64_t)a.W * a.K));
    float u[6];
    for (int l = 0; l < a.n_heads; ++l) {
      const int c = a.c[l];
      float s = 0.f;
      for (int ch = 0; ch < c; ++ch) s = fmaf(a.w1[l][(int64_t)ch * a.K + k], a.dg[l][(int64_t)b * a.W * c + w * c + ch], s);
      u[l] = s;
      a.U[(((int64_t)l * a.B + b) * a.K + k) * a.W + w] = s;
    }
    for (int h = 0; h < a.H; ++h) {
      float s = 0.f;
      for (int l = 0; l < a.n_heads; ++l) s = fmaf(a.w2[l][h], u[l], s);
      a.dfeat[(((int64_t)b * a.K + k) * a.H + h) * a.W + w] = s;
    }
  }
}

// P_l[b, k, w] = sum_h v_l[h] F[b, k, h, w] for all heads (the forward's height-reduced volume): one thread per (b, k, w)
template <typename T>
__global__ void heads_bwd_reduce_h_kernel(const HeadsBwdArgs a, float* __restrict__ P) {
  const int64_t total = (int64_t)a.B * a.K * a.W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % a.W);
    const int k = (int)((i / a.W) % a.K);
    const int b = (int)(i / ((int64_t)a.W * a.K));
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int h = 0; h < a.H; ++h) {
      const float f = feat_at<T>(a, b, k, h, w);
      for (int l = 0; l < a.n_heads; ++l) acc[l] = fmaf(a.w2[l][h], f, acc[l]);
    }
    for (int l = 0; l < a.n_heads; ++l) P[(((int64_t)l * a.B + b) * a.K + k) * a.W + w] = acc[l];
  }
}

// dW_l[ch, k] = sum_{b, w} dT_l[b, ch, w] * P_l[b, k, w]: one thread per (ch, k), B*W terms
__global__ void heads_bwd_w1_kernel(const HeadsBwdArgs a, const float* __restrict__ P, int l) {
  const int c = a.c[l];
  const int64_t total = (int64_t)c * a.K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % a.K), ch = (int)(i / a.K);
    float s = 0.f;
    for (int b = 0; b < a.B; ++b) {
      const float* pr = P + (((int64_t)l * a.B + b) * a.K + k) * a.W;
      const float* dr = a.dg[l] + (int64_t)b * a.W * c + ch;
      for (int w = 0; w < a.W; ++w) s = fmaf(dr[(int64_t)w * c], pr[w], s);
    }
    a.dw1[l][(int64_t)ch * a.K + k] = s;
  }
}

// dv_l[h] = sum_{b,k,w} F[b,k,h,w] U_l[b,k,w] (+ the b1 term, added by the small kernel): one block per (l, h)
template <typename T>
__global__ void __launch_bounds__(256) heads_bwd_w2_kernel(const HeadsBwdArgs a) {
  __shared__ float red[256];
  const int l = blockIdx.x, h = blockIdx.y, t = threadIdx.x;
  float s = 0.f;
  const int64_t total = (int64_t)a.B * a.K * a.W;
  for (int64_t i = t; i < total; i += 256) {
    const int w = (int)(i % a.W);
    const int k = (int)((i / a.W) % a.K);
    const int b = (int)(i / ((int64_t)a.W * a.K));
    s = fmaf(feat_at<T>(a, b, k, h, w), a.U[(((int64_t)l * a.B + b) * a.K + k) * a.W + w], s);
  }
  red[t] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {                 // fixed tree: deterministic
    if (t < o) red[t] += red[t + o];
    __syncthreads();
  }
  if (t == 0) a.dw2[l][h] = red[0];
}

// db1_l[ch], db2_l and the b1 term of dv_l: one block per head; thread-strided partials folded in a fixed order
// (runs AFTER heads_bwd_w2_kernel: it adds the b1 term to dw2)
__global__ void __launch_bounds__(256) heads_bwd_small_kernel(const HeadsBwdArgs a) {
  __shared__ float red[256];
  const int l = blockIdx.x;
  const int c = a.c[l];
  const int t = threadIdx.x;
  float vsum = 0.f;
  for (int h = 0; h < a.H; ++h) vsum += a.w2[l][h];
  for (int ch = 0; ch < c; ++ch) {
    float s = 0.f;
    for (int i = t; i < a.B * a.W; i += 256) {
      const int b = i / a.W, w = i - b * a.W;
      s += a.dg[l][(int64_t)b * a.W * c + w * c + ch];
    }
    red[t] = s;
    __syncthreads();
    if (t == 0) {
      float tot = 0.f;
      for (int i = 0; i < 256; ++i) tot += red[i];
      a.db1[l][ch] = tot * vsum;
    }
    __syncthreads();
  }
  float s_dg = 0.f, s_b1 = 0.f;
  for (int i = t; i < a.B * a.W * c; i += 256) {
    const float v = a.dg[l][i];
    s_dg += v;
    s_b1 = fmaf(v, a.b1[l][i % c], s_b1);
  }
  red[t] = s_dg;
  __syncthreads();
  if (t == 0) {
    float tot = 0.f;
    for (int i = 0; i < 256; ++i) tot += red[i];
    a.db2[l][0] = tot;
  }
  __syncthreads();
  red[t] = s_b1;
  __syncthreads();
  if (t == 0) {
    float x = 0.f;
    for (int i = 0; i < 256; ++i) x += red[i];
    for (int h = 0; h < a.H; ++h) a.dw2[l][h] += x;
  }
}

}  // namespace ccvpe

extern "C" int ccvpe_grd_descriptors_bwd(const void* feat, int dtype, int B, int K, int H, int W, int64_t sb, int64_t sk,
                                         int64_t sh, int64_t sw, int n_heads, const float* const* w1,
                                         const float* const* b1, const float* const* w2, const int32_t* c,
                                         const float* const* dg, float* dfeat, float* const* dw1, float* const* db1,
                                         float* const* dw2, float* const* db2, float* scratch, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(feat && w1 && b1 && w2 && c && dg && dfeat && dw1 && db1 && dw2 && db2 && scratch,
                "ccvpe_grd_descriptors_bwd: null pointer");
  CCVPE_REQUIRE(B > 0 && K > 0 && H > 0 && W > 0 && n_heads > 0 && n_heads <= 6, "ccvpe_grd_descriptors_bwd: bad shape");
  CCVPE_REQUIRE(dtype == CCVPE_F32 || dtype == CCVPE_BF16, "ccvpe_grd_descriptors_bwd: bad dtype");
  HeadsBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.feat = feat; a.dtype = dtype; a.B = B; a.K = K; a.H = H; a.W = W; a.sb = sb; a.sk = sk; a.sh = sh; a.sw = sw;
  a.n_heads = n_heads;
  for (int l = 0; l < n_heads; ++l) {
    a.w1[l] = w1[l]; a.b1[l] = b1[l]; a.w2[l] = w2[l]; a.dg[l] = dg[l]; a.c[l] = c[l];
    a.dw1[l] = dw1[l]; a.db1[l] = db1[l]; a.dw2[l] = dw2[l]; a.db2[l] = db2[l];
  }
  a.U = scratch;
  a.dfeat = dfeat;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ew_blocks((int64_t)B * K * W);
  if (dtype == CCVPE_F32) heads_bwd_data_kernel<float><<<blocks, 256, 0, st>>>(a);
  else heads_bwd_data_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(a);
  CCVPE_LAUNCH_CHECK("heads_bwd_data_kernel");
  float* P = scratch + (int64_t)n_heads * B * K * W;
  if (dtype == CCVPE_F32) heads_bwd_reduce_h_kernel<float><<<blocks, 256, 0, st>>>(a, P);
  else heads_bwd_reduce_h_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(a, P);
  CCVPE_LAUNCH_CHECK("heads_bwd_reduce_h_kernel");
  for (int l = 0; l < n_heads; ++l) {
    heads_bwd_w1_kernel<<<ew_blocks((int64_t)c[l] * K), 256, 0, st>>>(a, P, l);
    CCVPE_LAUNCH_CHECK("heads_bwd_w1_kernel");
  }
  if (dtype == CCVPE_F32) heads_bwd_w2_kernel<float><<<dim3(n_heads, H), 256, 0, st>>>(a);
  else heads_bwd_w2_kernel<__nv_bfloat16><<<dim3(n_heads, H), 256, 0, st>>>(a);
  CCVPE_LAUNCH_CHECK("heads_bwd_w2_kernel");
  heads_bwd_small_kernel<<<n_heads, 256, 0, st>>>(a);
  CCVPE_LAUNCH_CHECK("heads_bwd_small_kernel");
  return CCVPE_OK;
}
