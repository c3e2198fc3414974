// First step of SURVEY section 8(f)-2 (the PyTorch encoders are the end-to-end bottleneck once the decoder is fast):
// one fused, vectorised pass for the glue between the encoder's cuDNN/cuBLAS calls,
//
//   y[b, h, w, c] = SiLU( x[b, h, w, c] + bias[c] )          (+ optional per-(b, c) sum over h, w of y)
//
// x is a contiguous channels-last bf16 tensor; y may be a strided view (the interior of a pre-zeroed padded buffer, so
// the TensorFlow-"same" / circular padding of the following depthwise conv costs no extra copy); the channel sums feed
// the squeeze-excite gate, so the separate mean pass over the 6x-expanded activation disappears as well.
// HBM-bound: one read + one write of the tensor, 16-byte accesses.
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace ccvpe {

// Squeeze-excite channel sums are accumulated in 64-bit FIXED POINT (2^-20 units): integer addition is associative, so the
// result does not depend on the order in which threads and blocks arrive -- the bf16 path is bit-reproducible run to run
// (eager or CUDA-graph replay).  Every thread's own partial is a plain fp32 sum over a fixed set of pixels.  Head room:
// |sum| < 2^43 ~ 8.8e12, i.e. 65536 pixels of magnitude 1e8.
constexpr float kSeFixedScale = 1048576.f;
__device__ __forceinline__ unsigned long long se_fixed(float v) {
  return (unsigned long long)__float2ll_rn(v * kSeFixedScale);
}

__global__ void __launch_bounds__(256)
bias_silu_nhwc_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ bias,
                      __nv_bfloat16* __restrict__ y, int64_t y_sb, int64_t y_sh, int64_t y_sw, int H, int W, int C,
                      int pix_per_block, long long* __restrict__ chan_sum) {
  extern __shared__ unsigned long long s_sum[];    // [C] per-block channel sums, fixed point (only if chan_sum)
  const int G = C >> 3;                            // 8-channel groups per pixel
  const int lanes = blockDim.x / G;                // pixels processed concurrently by the block
  const int cg = threadIdx.x % G, pl = threadIdx.x / G;
  const int b = blockIdx.y;
  const int HW = H * W;
  const int p_lo = blockIdx.x * pix_per_block;
  const int p_hi = min(HW, p_lo + pix_per_block);
  if (chan_sum) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) s_sum[c] = 0ull;
    __syncthreads();
  }
  float bv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (bias && pl < lanes) {
    uint4 q = *reinterpret_cast<const uint4*>(bias + cg * 8);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 f = __bfloat1622float2(h[j]);
      bv[2 * j] = f.x;
      bv[2 * j + 1] = f.y;
    }
  }
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (pl < lanes) {
    const __nv_bfloat16* xb = x + (int64_t)b * HW * C + cg * 8;
    __nv_bfloat16* yb = y + (int64_t)b * y_sb + cg * 8;
    constexpr int U = 4;                           // independent 16-byte loads in flight per thread
    for (int p0 = p_lo + pl; p0 < p_hi; p0 += lanes * U) {
      uint4 q[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int p = p0 + u * lanes;
        if (p < p_hi) q[u] = __ldcs(reinterpret_cast<const uint4*>(xb + (int64_t)p * C));   // streamed: read once
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int p = p0 + u * lanes;
        if (p >= p_hi) break;
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q[u]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float2 f = __bfloat1622float2(h[j]);
          float a0 = f.x + bv[2 * j], a1 = f.y + bv[2 * j + 1];
          a0 = __fdividef(a0, 1.f + __expf(-a0));
          a1 = __fdividef(a1, 1.f + __expf(-a1));
          h[j] = __floats2bfloat162_rn(a0, a1);
          if (chan_sum) {                          // sum what is actually stored (bf16-rounded), like a mean of y
            float2 r = __bfloat1622float2(h[j]);
            acc[2 * j] += r.x;
            acc[2 * j + 1] += r.y;
          }
        }
        const int hh = p / W, ww = p - hh * W;
        *reinterpret_cast<uint4*>(yb + hh * y_sh + ww * y_sw) = q[u];
      }
    }
  }
  if (chan_sum) {
    if (pl < lanes) {
#pragma unroll
      for (int j = 0; j < 8; ++j) atomicAdd(&s_sum[cg * 8 + j], se_fixed(acc[j]));
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x)
      atomicAdd(reinterpret_cast<unsigned long long*>(chan_sum) + (int64_t)b * C + c, s_sum[c]);
  }
}

}  // namespace ccvpe

extern "C" int ccvpe_bias_silu_nhwc(const void* x, const void* bias, void* y, int64_t y_sb, int64_t y_sh, int64_t y_sw,
                                    int B, int H, int W, int C, int64_t* chan_sum, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && y, "ccvpe_bias_silu_nhwc: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0 && C <= 2048, "ccvpe_bias_silu_nhwc: bad shape B=%d H=%d W=%d C=%d",
                B, H, W, C);
  CCVPE_REQUIRE(aligned16(x) && aligned16(y) && aligned16(bias), "ccvpe_bias_silu_nhwc: pointers must be 16-byte aligned");
  CCVPE_REQUIRE(y_sw % 8 == 0 && y_sh % 8 == 0 && y_sb % 8 == 0, "ccvpe_bias_silu_nhwc: output strides must be multiples of 8");
  const int G = C / 8;
  CCVPE_REQUIRE(G <= 256, "ccvpe_bias_silu_nhwc: C too large");
  const int lanes = 256 / G;
  // enough blocks to fill the machine a few times over, each with a long pixel loop (few atomics per block)
  const int64_t HW = (int64_t)H * W;
  int blocks_x = (int)((8LL * sm_count() + B - 1) / B);
  int64_t ppb = (HW + blocks_x - 1) / blocks_x;
  ppb = (ppb + lanes - 1) / lanes * lanes;
  if (ppb < lanes) ppb = lanes;
  blocks_x = (int)((HW + ppb - 1) / ppb);
  bias_silu_nhwc_kernel<<<dim3(blocks_x, B), 256, chan_sum ? C * sizeof(unsigned long long) : 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)x, (const __nv_bfloat16*)bias, (__nv_bfloat16*)y, y_sb, y_sh, y_sw, H, W, C, (int)ppb, reinterpret_cast<long long*>(chan_sum));
  CCVPE_LAUNCH_CHECK("bias_silu_nhwc_kernel");
  return CCVPE_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Depthwise KxK convolution (stride 1 or 2) over a pre-padded channels-last buffer, fused with the folded-BN bias, SiLU
// and the squeeze-excite channel sums:
//     y[b, ho, wo, c] = SiLU( sum_{ky,kx} x[b, ho*S + ky, wo*S + kx, c] * w[ky, kx, c] + bias[c] ),   chan_sum[b, c] += y
// One thread owns 8 channels (16-byte vectors) and a strip of TW horizontally adjacent outputs, so every input vector is
// loaded once per strip and feeds up to K/S outputs per row; neighbouring strips share their halo through L1.
// Replaces cuDNN's depthwise conv + a separate bias/SiLU pass + a mean pass (reference model.py:108-114): one read of
// the padded input and one write of the activated output.  HBM-bound.
// ---------------------------------------------------------------------------------------------------------------------
namespace ccvpe {

// (packed fp32x2 helpers -- FFMA2 -- live in common.cuh: the loop below is issue-bound, so instruction count is what matters)
__device__ __forceinline__ float dw_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void dw_widen(const uint4& q, uint64_t (&f)[4]) {
  f[0] = bf16x2_to_f32x2(q.x);
  f[1] = bf16x2_to_f32x2(q.y);
  f[2] = bf16x2_to_f32x2(q.z);
  f[3] = bf16x2_to_f32x2(q.w);
}

// (measured: 4 channels per thread gains nothing over 8, the loop is issue-bound)
constexpr int DW_V = 8;                              // channels per thread: one 16-byte vector

template <int K, int S>
__global__ void __launch_bounds__(256, 2)
dwconv_bias_silu_kernel(const __nv_bfloat16* __restrict__ x, int64_t x_sb, int64_t x_sh, int64_t x_sw,
                        const __nv_bfloat16* __restrict__ w, const __nv_bfloat16* __restrict__ bias,
                        __nv_bfloat16* __restrict__ y, int Ho, int Wo, int C, int CG, int strips_per_block,
                        long long* __restrict__ chan_sum) {
  constexpr int V = DW_V;
  using vec_t = uint4;
  constexpr int P = V / 2;                           // fp32x2 pairs per thread
  constexpr int TW = 4;                              // outputs per thread along W
  constexpr int IW = (TW - 1) * S + K;               // input columns a strip touches
  // A block owns one image (blockIdx.y), one chunk of CG V-channel groups (blockIdx.z) and a range of strips
  // (blockIdx.x): wide low-resolution layers are split over channels so that every block still has a whole image's worth
  // of pixels to amortise its weight load over.
  // [lanes][CG*V] per-thread fp32 channel sums (folded in lane order at the end: no shared-memory atomics), then the
  // chunk's fp32 weights [K*K][CG*V]
  extern __shared__ __align__(16) float s_part[];
  const int CC = CG * V;                             // channels of a full chunk
  float* s_w = s_part + (blockDim.x / CG) * CC;
  const int G = C / V;
  const int g0 = blockIdx.z * CG;                    // first channel group of this chunk
  const int gn = min(CG, G - g0);                    // groups actually present in it
  const int lanes = blockDim.x / CG;
  const int cl = threadIdx.x % CG, pl = threadIdx.x / CG;
  const int cg = g0 + cl;
  const bool active = pl < lanes && cl < gn;
  const int b = blockIdx.y;
  {  // weight prologue: 4 channels per item, four independent loads in flight per thread (it is pure latency otherwise,
     // and the blocks of a wave all sit in it at the same time)
    const int q4 = gn * V / 4, n_items = K * K * q4;
#pragma unroll 1
    for (int i0 = threadIdx.x; i0 < n_items; i0 += 4 * blockDim.x) {
      uint2 v[4];
      int dst[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * blockDim.x;
        const int ii = i < n_items ? i : 0;
        const int tap = ii / q4, c4 = ii - tap * q4;
        v[u] = __ldg(reinterpret_cast<const uint2*>(w + (int64_t)tap * C + g0 * V) + c4);
        dst[u] = i < n_items ? tap * CC + c4 * 4 : -1;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (dst[u] >= 0)
          *reinterpret_cast<float4*>(s_w + dst[u]) =          // (pre-halved: the accumulator is h = a / 2 of the SiLU form)
              make_float4(0.5f * __uint_as_float(v[u].x << 16), 0.5f * __uint_as_float(v[u].x & 0xffff0000u),
                          0.5f * __uint_as_float(v[u].y << 16), 0.5f * __uint_as_float(v[u].y & 0xffff0000u));
    }
  }
  const int strips_row = (Wo + TW - 1) / TW;
  const int n_strips = Ho * strips_row;
  const int s_lo = blockIdx.x * strips_per_block;
  const int s_hi = min(n_strips, s_lo + strips_per_block);
  __syncthreads();
  float csum[V];
#pragma unroll
  for (int j = 0; j < V; ++j) csum[j] = 0.f;
  if (active) {
    uint64_t bv[P];
    dw_widen(*reinterpret_cast<const vec_t*>(bias + cg * V), bv);
#pragma unroll
    for (int j = 0; j < P; ++j) {                       // bias pre-halved like the weights
      float lo, hi;
      unpack_f32x2(bv[j], lo, hi);
      bv[j] = pack_f32x2(0.5f * lo, 0.5f * hi);
    }
    const __nv_bfloat16* xb = x + (int64_t)b * x_sb + cg * V;
    __nv_bfloat16* yb = y + (int64_t)b * Ho * Wo * C + cg * V;
    const float* wt = s_w + cl * V;
    // columns beyond the padded buffer can only feed outputs >= Wo (never stored): clamp them to stay in bounds
    const int iw_max = (Wo - 1) * S + K - 1;
    const int sw = (int)x_sw;                         // (32-bit offsets: one IMAD.WIDE per load address)
    for (int sidx = s_lo + pl; sidx < s_hi; sidx += lanes) {
      const int ho = sidx / strips_row;
      const int wo0 = (sidx - ho * strips_row) * TW;
      uint64_t acc[TW][P];
#pragma unroll
      for (int t = 0; t < TW; ++t)
#pragma unroll
        for (int j = 0; j < P; ++j) acc[t][j] = bv[j];
      const int ix_max = iw_max - wo0 * S;            // >= IW - 1 except on the right-most strip of a row
      const __nv_bfloat16* xrow = xb + (int64_t)(ho * S) * x_sh + (int64_t)(wo0 * S) * x_sw;
#pragma unroll 1
      for (int ky = 0; ky < K; ++ky, xrow += x_sh) {  // not unrolled: bounds the register footprint
        vec_t xin[IW];                                // the row segment this strip needs, still packed bf16
#pragma unroll
        for (int ix = 0; ix < IW; ++ix)
          xin[ix] = __ldg(reinterpret_cast<const vec_t*>(xrow + min(ix, ix_max) * sw));
        uint64_t xf[IW][P];                           // widened lazily: at most TW columns are live at a time
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
          uint64_t wv[P];
#pragma unroll
          for (int j = 0; j < P; j += 2) {
            const float4 wq = *reinterpret_cast<const float4*>(wt + (ky * K + kx) * CC + 2 * j);
            wv[j] = pack_f32x2(wq.x, wq.y);
            wv[j + 1] = pack_f32x2(wq.z, wq.w);
          }
#pragma unroll
          for (int t = 0; t < TW; ++t) {
            const int ix = t * S + kx;
            if (t == TW - 1 || kx < S) dw_widen(xin[ix], xf[ix]);      // first use of this input column
#pragma unroll
            for (int j = 0; j < P; ++j) acc[t][j] = ffma2(xf[ix][j], wv[j], acc[t][j]);
          }
        }
      }
#pragma unroll
      for (int t = 0; t < TW; ++t) {
        const int wo = wo0 + t;
        if (wo < Wo) {
          vec_t q;
          __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
          for (int j = 0; j < P; ++j) {
            float a0, a1;
            unpack_f32x2(acc[t][j], a0, a1);
            a0 = fmaf(a0, dw_tanh(a0), a0);           // SiLU(a) = a * sigmoid(a) = h + h * tanh(h), h = a / 2: one MUFU
            a1 = fmaf(a1, dw_tanh(a1), a1);
            h[j] = __floats2bfloat162_rn(a0, a1);
            const float2 r = __bfloat1622float2(h[j]);
            csum[2 * j] += r.x;
            csum[2 * j + 1] += r.y;
          }
          *reinterpret_cast<vec_t*>(yb + ((int64_t)ho * Wo + wo) * C) = q;
        }
      }
    }
  }
  if (chan_sum) {
    if (pl < lanes) {
#pragma unroll
      for (int j = 0; j < V; ++j) s_part[pl * CC + cl * V + j] = active ? csum[j] : 0.f;
    }
    __syncthreads();
    // one thread per channel folds the lanes in a fixed order (deterministic fp32), then ONE fixed-point atomic per
    // (block, channel) into the order-independent 64-bit accumulator
    for (int c = threadIdx.x; c < gn * V; c += blockDim.x) {
      float tot = 0.f;
      for (int l = 0; l < lanes; ++l) tot += s_part[l * CC + c];
      atomicAdd(reinterpret_cast<unsigned long long*>(chan_sum) + (int64_t)b * C + g0 * V + c, se_fixed(tot));
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Stride-1 depthwise convolution, shared-memory tiled version (same arithmetic and summation order as the kernel above,
// so y is bit-identical to it).  The streaming kernel above is bound by load latency at 128 registers per thread and
// by the LSU (every input vector is fetched K times, every fp32 weight vector once per four outputs); here
//   * a persistent CTA walks (image, 64-channel block, spatial tile) work items; the haloed input tile and the tile's
//     K*K x 64 bf16 weights arrive through cp.async into one of two stages, so the next item's loads are in flight during
//     the current item's arithmetic and cost no registers;
//   * a thread owns 4 channels (8-byte shared loads: the 16 lanes of a half warp read one pixel's 128 bytes, conflict
//     free) and a 2 x 8 output micro tile: (K+1) x (K+7) input vectors and K*K packed weights feed 16 outputs, i.e.
//     7.6 (5x5) shared loads per output instead of 22.5 -- the FMA pipe, not the LSU, is the limit.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int DWT_THREADS = 256;
constexpr int DWT_CB = 64;          // channels per work item
constexpr int DWT_PT = 16;          // pixel threads per work item (x 16 channel lanes = 256 threads)
constexpr int DWT_TW = 8, DWT_TH = 2;
constexpr int DWT_SCRATCH = DWT_PT * DWT_CB * 4;      // per-thread channel sums of one item
constexpr int DWT_STAGE_LIMIT = 55 * 1024;

struct DwTileParams {
  const __nv_bfloat16* x;
  int64_t x_sb, x_sh, x_sw;
  int Hp, Wp;
  const __nv_bfloat16* w;
  const __nv_bfloat16* bias;
  __nv_bfloat16* y;
  int Ho, Wo, C;
  int ptw, pth, otw, oth, itw, ith;
  int tiles_w, tiles_h, cblocks, total_items, stage_bytes;
  long long* chan_sum;
};

__device__ __forceinline__ void dwt_cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ uint2 dwt_lds64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}

template <int K>
__global__ void __launch_bounds__(DWT_THREADS, 2) dwconv_tile_kernel(const __grid_constant__ DwTileParams p) {
  constexpr int TW = DWT_TW, TH = DWT_TH, IW = TW + K - 1, IH = TH + K - 1;
  extern __shared__ __align__(128) uint8_t dwt_smem[];
  float* s_part = reinterpret_cast<float*>(dwt_smem);
  const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(dwt_smem) + DWT_SCRATCH;
  const int tid = threadIdx.x;
  const int cg = tid & 15, pt = tid >> 4;
  const int pw = pt % p.ptw, ph = pt / p.ptw;
  const int n_pix = p.ith * p.itw;

  auto decode = [&](int item, int& tw_i, int& th_i, int& cb, int& b) {
    tw_i = item % p.tiles_w;
    item /= p.tiles_w;
    th_i = item % p.tiles_h;
    item /= p.tiles_h;
    cb = item % p.cblocks;
    b = item / p.cblocks;
  };
  // loads of one work item: thread = (16-byte chunk of the pixel's 128 bytes, every 32nd pixel)
  auto issue = [&](int item, int stage) {
    int tw_i, th_i, cb, b;
    decode(item, tw_i, th_i, cb, b);
    const int c0 = cb * DWT_CB;
    const int nch = min(8, (p.C - c0) >> 3);
    const int ch = tid & 7;
    if (ch < nch) {
      const uint32_t sw = stage0 + (uint32_t)(stage * p.stage_bytes), sx = sw + K * K * 128;
      const __nv_bfloat16* xb = p.x + (int64_t)b * p.x_sb + c0 + ch * 8;
      const int gh0 = th_i * p.oth, gw0 = tw_i * p.otw;
      int pix = tid >> 3;
      int ih = pix / p.itw, iw = pix - ih * p.itw;
      for (; pix < n_pix; pix += 32) {
        // (rows / columns past the padded image only feed outputs that are never stored: clamp to stay in bounds)
        const int gh = min(gh0 + ih, p.Hp - 1), gw = min(gw0 + iw, p.Wp - 1);
        dwt_cp_async16(sx + (uint32_t)pix * 128u + (uint32_t)ch * 16u, xb + gh * p.x_sh + gw * p.x_sw);
        iw += 32;
        while (iw >= p.itw) {
          iw -= p.itw;
          ++ih;
        }
      }
      for (int tap = tid >> 3; tap < K * K; tap += 32)
        dwt_cp_async16(sw + (uint32_t)tap * 128u + (uint32_t)ch * 16u, p.w + (int64_t)tap * p.C + c0 + ch * 8);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  int item = blockIdx.x;
  if (item < p.total_items) issue(item, 0);
  for (int it = 0; item < p.total_items; item += gridDim.x, ++it) {
    const int nxt = item + gridDim.x;
    if (nxt < p.total_items) {
      issue(nxt, (it + 1) & 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    int tw_i, th_i, cb, b;
    decode(item, tw_i, th_i, cb, b);
    const int c0 = cb * DWT_CB;
    const bool active = (c0 + cg * 4 < p.C) && ph < p.pth;
    float csum[4] = {0.f, 0.f, 0.f, 0.f};
    if (active) {
      const uint32_t sw = stage0 + (uint32_t)((it & 1) * p.stage_bytes) + (uint32_t)cg * 8u;
      const uint32_t sx = sw + K * K * 128 + (uint32_t)((ph * TH) * p.itw + pw * TW) * 128u;
      const uint32_t row_pitch = (uint32_t)p.itw * 128u;
      uint64_t bv[2];
      {
        const uint2 bq = __ldg(reinterpret_cast<const uint2*>(p.bias + c0 + cg * 4));
        bv[0] = bf16x2_to_f32x2(bq.x);
        bv[1] = bf16x2_to_f32x2(bq.y);
      }
      uint64_t acc[TH][TW][2];
#pragma unroll
      for (int r = 0; r < TH; ++r)
#pragma unroll
        for (int t = 0; t < TW; ++t) {
          acc[r][t][0] = bv[0];
          acc[r][t][1] = bv[1];
        }
#pragma unroll
      for (int ir = 0; ir < IH; ++ir) {
        uint2 xin[IW];
#pragma unroll
        for (int ix = 0; ix < IW; ++ix) xin[ix] = dwt_lds64(sx + (uint32_t)ir * row_pitch + (uint32_t)ix * 128u);
        uint64_t xf[IW][2];
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
#pragma unroll
          for (int t = 0; t < TW; ++t)
            if (kx == 0 || t == TW - 1) {              // first use of input column t + kx
              xf[t + kx][0] = bf16x2_to_f32x2(xin[t + kx].x);
              xf[t + kx][1] = bf16x2_to_f32x2(xin[t + kx].y);
            }
#pragma unroll
          for (int r = 0; r < TH; ++r) {
            const int ky = ir - r;                     // input row ir is row ky of output row r's window
            if (ky >= 0 && ky < K) {
              const uint2 wq = dwt_lds64(sw + (uint32_t)(ky * K + kx) * 128u);
              const uint64_t w0 = bf16x2_to_f32x2(wq.x), w1 = bf16x2_to_f32x2(wq.y);
#pragma unroll
              for (int t = 0; t < TW; ++t) {
                acc[r][t][0] = ffma2(xf[t + kx][0], w0, acc[r][t][0]);
                acc[r][t][1] = ffma2(xf[t + kx][1], w1, acc[r][t][1]);
              }
            }
          }
        }
      }
      const int ho0 = th_i * p.oth + ph * TH, wo0 = tw_i * p.otw + pw * TW;
#pragma unroll
      for (int r = 0; r < TH; ++r) {
        const int ho = ho0 + r;
        if (ho < p.Ho) {
          __nv_bfloat16* yrow = p.y + (((int64_t)b * p.Ho + ho) * p.Wo) * p.C + c0 + cg * 4;
#pragma unroll
          for (int t = 0; t < TW; ++t) {
            const int wo = wo0 + t;
            if (wo < p.Wo) {
              uint2 q;
              __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                float a0, a1;
                unpack_f32x2(acc[r][t][j], a0, a1);
                a0 *= 0.5f;                             // SiLU(a) = h + h * tanh(h), h = a / 2 (one MUFU)
                a1 *= 0.5f;
                a0 = fmaf(a0, dw_tanh(a0), a0);
                a1 = fmaf(a1, dw_tanh(a1), a1);
                h[j] = __floats2bfloat162_rn(a0, a1);
                const float2 rr = __bfloat1622float2(h[j]);
                csum[2 * j] += rr.x;
                csum[2 * j + 1] += rr.y;
              }
              *reinterpret_cast<uint2*>(yrow + (int64_t)wo * p.C) = q;
            }
          }
        }
      }
    }
    if (p.chan_sum) {
#pragma unroll
      for (int j = 0; j < 4; ++j) s_part[pt * DWT_CB + cg * 4 + j] = csum[j];
    }
    __syncthreads();   // the stage is free for the item after next; the per-thread sums are visible
    if (p.chan_sum && tid < DWT_CB && c0 + tid < p.C) {
      // fixed-order fp32 fold of the 16 pixel threads, then one order-independent fixed-point atomic per (item, channel)
      float tot = 0.f;
#pragma unroll
      for (int l = 0; l < DWT_PT; ++l) tot += s_part[l * DWT_CB + tid];
      atomicAdd(reinterpret_cast<unsigned long long*>(p.chan_sum) + (int64_t)b * p.C + c0 + tid, se_fixed(tot));
    }
  }
}

// picks the micro-tile arrangement (ptw x pth pixel threads, each 2 rows x 8 columns) of the tiled kernel; false if no
// arrangement fits the stage budget
static bool dwt_plan(int K, int Ho, int Wo, int C, int B, DwTileParams* p) {
  double best = 1e30;
  bool found = false;
  for (int ptw = 1; ptw <= DWT_PT; ++ptw) {
    const int pth = DWT_PT / ptw;
    const int otw = ptw * DWT_TW, oth = pth * DWT_TH;
    const int itw = otw + K - 1, ith = oth + K - 1;
    const int stage = (K * K + ith * itw) * 128;
    if (stage > DWT_STAGE_LIMIT) continue;
    const int tiles_w = (Wo + otw - 1) / otw, tiles_h = (Ho + oth - 1) / oth;
    // cost of the layer ~ items x (bytes staged + the fixed arithmetic of a full item)
    const double cost = (double)tiles_w * tiles_h * (ith * itw + 2.0 * DWT_PT * DWT_TW * DWT_TH);
    if (cost < best) {
      best = cost;
      found = true;
      p->ptw = ptw; p->pth = pth; p->otw = otw; p->oth = oth; p->itw = itw; p->ith = ith;
      p->tiles_w = tiles_w; p->tiles_h = tiles_h; p->stage_bytes = stage;
    }
  }
  if (!found) return false;
  p->cblocks = (C + DWT_CB - 1) / DWT_CB;
  const int64_t total = (int64_t)p->tiles_w * p->tiles_h * p->cblocks * B;
  if (total > (1LL << 30)) return false;
  p->total_items = (int)total;
  return true;
}

// The depthwise dispatch, shared by the launch and by ccvpe_dwconv_plan so that the two cannot disagree: checks the shape,
// then returns 1 for dwconv_tile_kernel (its plan in *tp), 0 for dwconv_bias_silu_kernel, < 0 on a bad argument.
// Measured per layer (B=64, scripts/bench_dwconv.py): the tiled kernel wins wherever the window is 5x5 (1.2-1.5x) and for
// the deep 3x3 layers (>= 240 channels); the shallow 3x3 layers (32 / 144 channels on large images) and every stride-2
// layer stay on the streaming kernel.
static int dw_select(int B, int C, int Hp, int Wp, int K, int S, DwTileParams* tp) {
  CCVPE_REQUIRE(B > 0 && C > 0 && C % 8 == 0 && C <= 2048, "ccvpe_dwconv_bias_silu_nhwc: bad shape B=%d C=%d", B, C);
  CCVPE_REQUIRE((K == 3 || K == 5) && (S == 1 || S == 2) && Hp >= K && Wp >= K, "ccvpe_dwconv_bias_silu_nhwc: K=%d S=%d Hp=%d Wp=%d unsupported", K, S, Hp, Wp);
  const int Ho = (Hp - K) / S + 1, Wo = (Wp - K) / S + 1;
  memset(tp, 0, sizeof(*tp));
  if (S == 1 && (K == 5 || C >= 240) && dwt_plan(K, Ho, Wo, C, B, tp)) return 1;
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Encoder stem: see stem_tcgen05.cu (3x3 stride-2 convolution over the planar fp32 / uint8 image as an implicit GEMM on the
// tensor cores + folded-BN bias + SiLU, written as bf16 channels-last into the interior of the first depthwise
// convolution's padded input image, wrap columns included for the circular encoder).  The CUDA-core kernel that used to
// live here (864 packed FMAs per pixel pair, 0.29 + 0.32 ms per step) was retired in round 2.
// ---------------------------------------------------------------------------------------------------------------------
// Squeeze-excite gate folded into the projection weights, one launch per MBConv block:
//     mean[b, m]   = chan_sum[b, m] * inv_hw
//     h[b, r]      = SiLU(b_red[r] + sum_m w_red[r, m] * mean[b, m])
//     g[b, m]      = sigmoid(b_se[m] + sum_r w_se_t[r, m] * h[b, r])      (w_se_t = transposed excite weights)
//     wg[b, c, m]  = w_proj[c, m] * g[b, m]                (the B operand of the per-image projection GEMM)
// Replaces seven small PyTorch launches per block (div, cast, two addmm, silu, sigmoid, mul).  fp32 math, bf16 in / out.
// grid (B, row chunks): every block recomputes its image's gate (two tiny mat-vecs) and scales its rows of w_proj.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512)
se_gate_scale_kernel(const long long* __restrict__ chan_sum, float inv_hw, const __nv_bfloat16* __restrict__ w_red,
                     const __nv_bfloat16* __restrict__ b_red, const __nv_bfloat16* __restrict__ w_se_t,
                     const __nv_bfloat16* __restrict__ b_se, const __nv_bfloat16* __restrict__ w_proj,
                     __nv_bfloat16* __restrict__ wg, int mid, int R, int cout, int rows_per_block) {
  extern __shared__ __align__(16) float s_se[];      // mean[mid] (later g[mid]), h[R]
  float* s_mean = s_se;
  float* s_h = s_se + mid;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int m = tid; m < mid; m += blockDim.x) s_mean[m] = __ll2float_rn(chan_sum[(int64_t)b * mid + m]) * (inv_hw * (1.f / kSeFixedScale));
  __syncthreads();
  const int n_warps = blockDim.x >> 5;
  for (int r = warp; r < R; r += n_warps) {           // one warp per reduced channel, 8 bf16 per lane per step
    const __nv_bfloat16* wr = w_red + (int64_t)r * mid;
    float acc = 0.f;
    for (int m0 = lane * 8; m0 < mid; m0 += 256) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(wr + m0));
      const __nv_bfloat162* hq = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(hq[j]);
        acc = fmaf(f.x, s_mean[m0 + 2 * j], acc);
        acc = fmaf(f.y, s_mean[m0 + 2 * j + 1], acc);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const float v = acc + __bfloat162float(b_red[r]);
      s_h[r] = __fdividef(v, 1.f + __expf(-v));
    }
  }
  __syncthreads();
  for (int m = tid; m < mid; m += blockDim.x) {       // gate: one channel per thread, R (<= 48) terms, coalesced over m
    float acc = __bfloat162float(b_se[m]);
#pragma unroll 8
    for (int r = 0; r < R; ++r) acc = fmaf(__bfloat162float(__ldg(w_se_t + (int64_t)r * mid + m)), s_h[r], acc);
    s_mean[m] = __fdividef(1.f, 1.f + __expf(-acc));  // (each thread overwrites only the means it owns)
  }
  __syncthreads();
  const int c_lo = blockIdx.y * rows_per_block, c_hi = min(cout, c_lo + rows_per_block);
  const int vec_per_row = mid >> 3;
  const int total = (c_hi - c_lo) * vec_per_row;
  const uint4* src = reinterpret_cast<const uint4*>(w_proj + (int64_t)c_lo * mid);
  uint4* dst = reinterpret_cast<uint4*>(wg + ((int64_t)b * cout + c_lo) * mid);
  for (int i = tid; i < total; i += blockDim.x) {
    const int m0 = (i % vec_per_row) * 8;
    uint4 q = __ldg(src + i);
    __nv_bfloat162* hq = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(hq[j]);
      hq[j] = __floats2bfloat162_rn(f.x * s_mean[m0 + 2 * j], f.y * s_mean[m0 + 2 * j + 1]);
    }
    dst[i] = q;
  }
}

// Two-kernel form of the same operator for the deep blocks (measured: the fused kernel spends 42 us per launch at
// mid = 1152 -- every block first recomputes the gate, a chain of dependent L2 loads, before it may scale its rows):
// se_gate_kernel computes g[b, :] once per image, se_scale_kernel is a flat grid-stride pass over all of wg.  `rep` > 1
// writes the block-diagonal weights of `rep` pixels packed into one GEMM row,
//   wg[b][r * cout + c][r' * mid + m] = (r == r') ? w_proj[c][m] * g[b][m] : 0,
// which lets the projection GEMM of the shallow first block (mid = 32: 64-byte pixels) read full 128-byte rows.
__global__ void __launch_bounds__(1024)
se_gate_kernel(const long long* __restrict__ chan_sum, float inv_hw, const __nv_bfloat16* __restrict__ w_red,
               const __nv_bfloat16* __restrict__ b_red, const __nv_bfloat16* __restrict__ w_se_t,
               const __nv_bfloat16* __restrict__ b_se, float* __restrict__ gate, int mid, int R) {
  extern __shared__ __align__(16) float s_se[];
  float* s_mean = s_se;
  float* s_h = s_se + mid;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int m = tid; m < mid; m += blockDim.x) s_mean[m] = __ll2float_rn(chan_sum[(int64_t)b * mid + m]) * (inv_hw * (1.f / kSeFixedScale));
  __syncthreads();
  const int n_warps = blockDim.x >> 5;
  for (int r = warp; r < R; r += n_warps) {
    const __nv_bfloat16* wr = w_red + (int64_t)r * mid;
    float acc = 0.f;
    for (int m0 = lane * 8; m0 < mid; m0 += 256) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(wr + m0));
      const __nv_bfloat162* hq = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(hq[j]);
        acc = fmaf(f.x, s_mean[m0 + 2 * j], acc);
        acc = fmaf(f.y, s_mean[m0 + 2 * j + 1], acc);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const float v = acc + __bfloat162float(b_red[r]);
      s_h[r] = __fdividef(v, 1.f + __expf(-v));
    }
  }
  __syncthreads();
  for (int m = tid; m < mid; m += blockDim.x) {
    float acc = __bfloat162float(b_se[m]);
#pragma unroll 8
    for (int r = 0; r < R; ++r) acc = fmaf(__bfloat162float(__ldg(w_se_t + (int64_t)r * mid + m)), s_h[r], acc);
    gate[(int64_t)b * mid + m] = __fdividef(1.f, 1.f + __expf(-acc));
  }
}

__global__ void __launch_bounds__(256)
se_scale_kernel(const float* __restrict__ gate, const __nv_bfloat16* __restrict__ w_proj, __nv_bfloat16* __restrict__ wg,
                int mid, int cout, int rep, int64_t total_vec) {
  const int row_vec = rep * mid >> 3;                       // 8-element vectors per output row
  const int64_t per_img = (int64_t)rep * cout * row_vec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total_vec; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / per_img);
    const int rem = (int)(i - (int64_t)b * per_img);
    const int row = rem / row_vec, k0 = (rem - row * row_vec) << 3;
    const int r = row / cout, c = row - r * cout;
    const int r2 = k0 / mid, m0 = k0 - r2 * mid;            // mid % 8 == 0: a vector never straddles two pixels
    uint4 q = make_uint4(0u, 0u, 0u, 0u);
    if (r == r2) {
      q = __ldg(reinterpret_cast<const uint4*>(w_proj + (int64_t)c * mid + m0));
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gate + (int64_t)b * mid + m0));
      const float4 g1 = __ldg(reinterpret_cast<const float4*>(gate + (int64_t)b * mid + m0 + 4));
      const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      __nv_bfloat162* hq = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __bfloat1622float2(hq[j]);
        hq[j] = __floats2bfloat162_rn(f.x * gv[2 * j], f.y * gv[2 * j + 1]);
      }
    }
    reinterpret_cast<uint4*>(wg)[i] = q;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Circular width padding of a padded channels-last image [B, Hp, Wp, C] whose interior (rows lo .. lo+H-1, columns
// lo .. lo+W-1) has been written: columns [0, lo) <- interior columns [W - lo, W), columns [lo + W, Wp) <- interior
// columns [0, hi).  One launch instead of two strided tensor copies per depthwise conv of the panorama encoder.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
wrap_columns_kernel(__nv_bfloat16* __restrict__ buf, int H, int W, int C, int lo, int hi, int Hp, int Wp, int64_t total) {
  const int vec = C >> 3;                                     // 16-byte vectors per pixel
  const int per_row = (lo + hi) * vec;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / per_row;                          // (b, h) of an interior row
    const int r = (int)(i - row * per_row);
    const int col = r / vec, v = r - col * vec;               // wrap column index 0 .. lo+hi-1
    const int b = (int)(row / H), h = (int)(row - (int64_t)b * H);
    const int dst_col = col < lo ? col : W + col;             // left wraps, then right wraps (padded coordinates)
    const int src_col = col < lo ? W + col : col;             // = dst_col +- W
    uint4* base = reinterpret_cast<uint4*>(buf + (((int64_t)b * Hp + h + lo) * Wp) * C);
    base[(int64_t)dst_col * vec + v] = base[(int64_t)src_col * vec + v];
  }
}

int igemm_tcgen05(const ccvpe_igemm_desc& d, cudaStream_t st, const TcOutPad* out_pad);  // igemm_tcgen05.cu

}  // namespace ccvpe

extern "C" int ccvpe_wrap_columns_nhwc(void* buf, int B, int H, int W, int C, int pad_lo, int pad_hi, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(buf && aligned16(buf), "ccvpe_wrap_columns_nhwc: buf must be a 16-byte aligned pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "ccvpe_wrap_columns_nhwc: bad shape");
  CCVPE_REQUIRE(pad_lo >= 0 && pad_hi >= 0 && pad_lo <= W && pad_hi <= W, "ccvpe_wrap_columns_nhwc: wrap wider than the image");
  if (pad_lo + pad_hi == 0) return CCVPE_OK;
  const int Hp = H + pad_lo + pad_hi, Wp = W + pad_lo + pad_hi;
  const int64_t total = (int64_t)B * H * (pad_lo + pad_hi) * (C / 8);
  int64_t blocks = (total + 255) / 256;
  if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
  wrap_columns_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)buf, H, W, C, pad_lo, pad_hi, Hp, Wp, total);
  CCVPE_LAUNCH_CHECK("wrap_columns_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_se_gate_scale(const int64_t* chan_sum, float inv_hw, const void* w_red, const void* b_red,
                                   const void* w_se, const void* b_se, const void* w_proj, void* wg, int B, int mid,
                                   int R, int cout, int rep, float* gate_ws, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(chan_sum && w_red && b_red && w_se && b_se && w_proj && wg, "ccvpe_se_gate_scale: null pointer");
  CCVPE_REQUIRE(B > 0 && B <= 65535 * 32 && mid > 0 && mid % 8 == 0 && R > 0 && cout > 0,
                "ccvpe_se_gate_scale: bad shape B=%d mid=%d R=%d cout=%d", B, mid, R, cout);
  CCVPE_REQUIRE(aligned16(w_red) && aligned16(w_proj) && aligned16(wg), "ccvpe_se_gate_scale: pointers must be 16-byte aligned");
  CCVPE_REQUIRE(rep >= 1 && rep <= 8, "ccvpe_se_gate_scale: rep=%d out of range", rep);
  CCVPE_REQUIRE(rep == 1 || gate_ws, "ccvpe_se_gate_scale: packed weights (rep > 1) need the gate workspace");
  CCVPE_REQUIRE((size_t)(mid + R) * sizeof(float) <= 48 * 1024, "ccvpe_se_gate_scale: mid too large");
  if (gate_ws && (rep > 1 || (int64_t)cout * mid >= 32768)) {
    CCVPE_REQUIRE(aligned16(gate_ws), "ccvpe_se_gate_scale: gate workspace must be 16-byte aligned");
    // (one block per image: both mat-vecs are chains of dependent L2 loads, so more threads = fewer rounds)
    se_gate_kernel<<<B, mid >= 512 ? 1024 : 512, (size_t)(mid + R) * sizeof(float), (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(chan_sum), inv_hw, (const __nv_bfloat16*)w_red, (const __nv_bfloat16*)b_red,
        (const __nv_bfloat16*)w_se, (const __nv_bfloat16*)b_se, gate_ws, mid, R);
    CCVPE_LAUNCH_CHECK("se_gate_kernel");
    const int64_t total_vec = (int64_t)B * rep * cout * (rep * mid / 8);
    int64_t blocks = (total_vec + 255) / 256;
    if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
    se_scale_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(gate_ws, (const __nv_bfloat16*)w_proj, (__nv_bfloat16*)wg, mid,
                                                                         cout, rep, total_vec);
    CCVPE_LAUNCH_CHECK("se_scale_kernel");
    return CCVPE_OK;
  }
  int rows = 98304 / mid;
  if (rows < 8) rows = 8;
  if (rows > cout) rows = cout;
  const dim3 grid(B, (cout + rows - 1) / rows);
  const size_t sm = (size_t)(mid + R) * sizeof(float);
  CCVPE_REQUIRE(sm <= 48 * 1024, "ccvpe_se_gate_scale: mid too large");
  se_gate_scale_kernel<<<grid, 512, sm, (cudaStream_t)stream>>>(
      reinterpret_cast<const long long*>(chan_sum), inv_hw, (const __nv_bfloat16*)w_red, (const __nv_bfloat16*)b_red, (const __nv_bfloat16*)w_se,
      (const __nv_bfloat16*)b_se, (const __nv_bfloat16*)w_proj, (__nv_bfloat16*)wg, mid, R, cout, rows);
  CCVPE_LAUNCH_CHECK("se_gate_scale_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_stem_conv_silu_nhwc(const float* x, int B, int H, int W, const float* w, const float* bias, int CO,
                                         void* out, int in_pad_lo, int in_pad_hi, int out_pad_lo, int out_pad_hi,
                                         int circular, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && w && bias && out, "ccvpe_stem_conv_silu_nhwc: null pointer");
  CCVPE_REQUIRE(B > 0 && H >= 3 && W >= 3 && B <= 65535, "ccvpe_stem_conv_silu_nhwc: bad shape B=%d H=%d W=%d", B, H, W);
  CCVPE_REQUIRE(CO == 32, "ccvpe_stem_conv_silu_nhwc: CO=%d unsupported (EfficientNet-B0 stem has 32 channels)", CO);
  CCVPE_REQUIRE(in_pad_lo >= 0 && in_pad_lo <= 2 && in_pad_hi >= 0 && in_pad_hi <= 2 && out_pad_lo >= 0 && out_pad_hi >= 0,
                "ccvpe_stem_conv_silu_nhwc: bad padding");
  CCVPE_REQUIRE(aligned16(out), "ccvpe_stem_conv_silu_nhwc: out must be 16-byte aligned");
  const int Ho = (H + in_pad_lo + in_pad_hi - 3) / 2 + 1, Wo = (W + in_pad_lo + in_pad_hi - 3) / 2 + 1;
  CCVPE_REQUIRE(!circular || (out_pad_lo <= Wo && out_pad_hi <= Wo), "ccvpe_stem_conv_silu_nhwc: wrap wider than the image");
  const int Hp = Ho + out_pad_lo + out_pad_hi, Wp = Wo + out_pad_lo + out_pad_hi;
  cudaStream_t st = (cudaStream_t)stream;
  StemTcParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.x = x; tp.w = w; tp.bias = bias; tp.out = (__nv_bfloat16*)out;
  tp.B = B; tp.H = H; tp.W = W; tp.Ho = Ho; tp.Wo = Wo; tp.in_lo = in_pad_lo; tp.out_lo = out_pad_lo; tp.Hp = Hp; tp.Wp = Wp;
  return stem_tcgen05(tp, circular != 0, false, st);
}

extern "C" int ccvpe_stem_conv_silu_u8_nhwc(const uint8_t* x, int B, int H, int Wsrc, int crop_w, const int32_t* shift,
                                            const float* mean_host, const float* std_host, const float* w, const float* bias,
                                            int CO, void* out, int in_pad_lo, int in_pad_hi, int out_pad_lo, int out_pad_hi,
                                            int circular, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && w && bias && out && mean_host && std_host, "ccvpe_stem_conv_silu_u8_nhwc: null pointer");
  const int W = crop_w;
  CCVPE_REQUIRE(B > 0 && H >= 3 && W >= 3 && W <= Wsrc && B <= 65535, "ccvpe_stem_conv_silu_u8_nhwc: bad shape B=%d H=%d W=%d Wsrc=%d",
                B, H, W, Wsrc);
  CCVPE_REQUIRE(CO == 32, "ccvpe_stem_conv_silu_u8_nhwc: CO=%d unsupported (EfficientNet-B0 stem has 32 channels)", CO);
  CCVPE_REQUIRE(in_pad_lo >= 0 && in_pad_lo <= 2 && in_pad_hi >= 0 && in_pad_hi <= 2 && out_pad_lo >= 0 && out_pad_hi >= 0,
                "ccvpe_stem_conv_silu_u8_nhwc: bad padding");
  CCVPE_REQUIRE(aligned16(out), "ccvpe_stem_conv_silu_u8_nhwc: out must be 16-byte aligned");
  const int Ho = (H + in_pad_lo + in_pad_hi - 3) / 2 + 1, Wo = (W + in_pad_lo + in_pad_hi - 3) / 2 + 1;
  CCVPE_REQUIRE(!circular || (out_pad_lo <= Wo && out_pad_hi <= Wo), "ccvpe_stem_conv_silu_u8_nhwc: wrap wider than the image");
  const int Hp = Ho + out_pad_lo + out_pad_hi, Wp = Wo + out_pad_lo + out_pad_hi;
  StemTcParams tp;
  memset(&tp, 0, sizeof(tp));
  tp.x8 = x; tp.shift = shift; tp.Wsrc = Wsrc;
  for (int c = 0; c < 3; ++c) {           // (u8 / 255 - mean) / std  ==  u8 * sc + sh
    tp.sc[c] = 1.f / (255.f * std_host[c]);
    tp.sh[c] = -mean_host[c] / std_host[c];
  }
  tp.w = w; tp.bias = bias; tp.out = (__nv_bfloat16*)out;
  tp.B = B; tp.H = H; tp.W = W; tp.Ho = Ho; tp.Wo = Wo; tp.in_lo = in_pad_lo; tp.out_lo = out_pad_lo; tp.Hp = Hp; tp.Wp = Wp;
  return stem_tcgen05(tp, circular != 0, true, (cudaStream_t)stream);
}

extern "C" int ccvpe_pointwise_silu_nhwc(const void* x, int B, int H, int W, int K, int ldx, const void* w_nk,
                                         const float* bias, int N, void* out, int pad_lo, int pad_hi, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && w_nk && out, "ccvpe_pointwise_silu_nhwc: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && (int64_t)B * H * W < (1LL << 31) - 256, "ccvpe_pointwise_silu_nhwc: bad shape");
  CCVPE_REQUIRE(K > 0 && K % 8 == 0 && N > 0 && N % 8 == 0 && ldx >= K && ldx % 8 == 0,
                "ccvpe_pointwise_silu_nhwc: K=%d N=%d ldx=%d must be positive multiples of 8", K, N, ldx);
  CCVPE_REQUIRE(pad_lo >= 0 && pad_hi >= 0, "ccvpe_pointwise_silu_nhwc: negative padding");
  CCVPE_REQUIRE(aligned16(x) && aligned16(w_nk) && aligned16(out), "ccvpe_pointwise_silu_nhwc: pointers must be 16-byte aligned");
  ccvpe_igemm_desc d;
  memset(&d, 0, sizeof(d));
  d.a0 = x; d.c0 = K; d.ld0 = ldx;
  d.B = B; d.Hin = d.Hout = H; d.Win = d.Wout = W;
  d.stride = 1; d.kh = d.kw = 1; d.pad = 0;
  d.N = N; d.dtype = CCVPE_BF16; d.w_nk = w_nk; d.bias = bias;
  d.relu = 2;                                   // SiLU epilogue
  d.out_mode = 0; d.out_dtype = CCVPE_BF16; d.ldo = N; d.out = out;
  d.backend = CCVPE_BACKEND_TCGEN05;
  const TcOutPad padded = {H + pad_lo + pad_hi, W + pad_lo + pad_hi, pad_lo};
  return igemm_tcgen05(d, (cudaStream_t)stream, (pad_lo || pad_hi) ? &padded : nullptr);
}

extern "C" int ccvpe_dwconv_bias_silu_nhwc(const void* x, int64_t x_sb, int64_t x_sh, int64_t x_sw, int Hp, int Wp,
                                           const void* w, const void* bias, void* y, int B, int C, int K, int S,
                                           int64_t* chan_sum, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(x && w && bias && y, "ccvpe_dwconv_bias_silu_nhwc: null pointer");
  DwTileParams tp;
  const int kernel = dw_select(B, C, Hp, Wp, K, S, &tp);
  if (kernel < 0) return kernel;
  CCVPE_REQUIRE(aligned16(x) && aligned16(w) && aligned16(bias) && aligned16(y), "ccvpe_dwconv_bias_silu_nhwc: pointers must be 16-byte aligned");
  CCVPE_REQUIRE(x_sb % 8 == 0 && x_sh % 8 == 0 && x_sw % 8 == 0, "ccvpe_dwconv_bias_silu_nhwc: input strides must be multiples of 8");
  CCVPE_REQUIRE(x_sw > 0 && x_sw * 16 < (1LL << 31), "ccvpe_dwconv_bias_silu_nhwc: pixel stride out of range");
  const int Ho = (Hp - K) / S + 1, Wo = (Wp - K) / S + 1;
  if (kernel == 1) {
    tp.x = (const __nv_bfloat16*)x; tp.x_sb = x_sb; tp.x_sh = x_sh; tp.x_sw = x_sw; tp.Hp = Hp; tp.Wp = Wp;
    tp.w = (const __nv_bfloat16*)w; tp.bias = (const __nv_bfloat16*)bias; tp.y = (__nv_bfloat16*)y;
    tp.Ho = Ho; tp.Wo = Wo; tp.C = C;
    tp.chan_sum = reinterpret_cast<long long*>(chan_sum);
    const int smem = DWT_SCRATCH + 2 * tp.stage_bytes;
    static thread_local uint64_t tiled_attr = 0;
    if (first_use_on_device(tiled_attr)) {
      cudaFuncSetAttribute(dwconv_tile_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, DWT_SCRATCH + 2 * DWT_STAGE_LIMIT);
      cudaFuncSetAttribute(dwconv_tile_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, DWT_SCRATCH + 2 * DWT_STAGE_LIMIT);
    }
    const int max_grid = 2 * sm_count();
    const int grid = tp.total_items < max_grid ? tp.total_items : max_grid;
    if (K == 3) dwconv_tile_kernel<3><<<grid, DWT_THREADS, smem, (cudaStream_t)stream>>>(tp);
    else dwconv_tile_kernel<5><<<grid, DWT_THREADS, smem, (cudaStream_t)stream>>>(tp);
    CCVPE_LAUNCH_CHECK("dwconv_tile_kernel");
    return CCVPE_OK;
  }
  constexpr int V = DW_V;
  const int G = C / V;
  // channel chunking: up to 256 channels a block takes them all; wider layers are cut into chunks of CG groups, CG the
  // largest divisor of G giving 64..128 channels (else 128 with a partial last chunk), which multiplies the number of
  // blocks on the low-resolution layers and keeps a block's weight tile small
  int CG = G;
  if (C > 256) {
    CG = 128 / V;
    for (int c = 128 / V; c >= 64 / V; --c)
      if (G % c == 0) {
        CG = c;
        break;
      }
  }
  const int chunks = (G + CG - 1) / CG;
  const int lanes = 256 / CG;
  const int64_t n_strips = (int64_t)Ho * ((Wo + 3) / 4);
  int blocks_x = (int)((8LL * sm_count() + (int64_t)B * chunks - 1) / ((int64_t)B * chunks));
  int64_t spb = (n_strips + blocks_x - 1) / blocks_x;
  spb = (spb + lanes - 1) / lanes * lanes;
  if (spb < lanes) spb = lanes;
  blocks_x = (int)((n_strips + spb - 1) / spb);
  CCVPE_REQUIRE(chunks <= 65535 && B <= 65535, "ccvpe_dwconv_bias_silu_nhwc: grid too large");
  const dim3 grid(blocks_x, B, chunks);
  const size_t sm = (size_t)CG * V * sizeof(float) * (lanes + K * K);
  CCVPE_REQUIRE(sm <= 96 * 1024, "ccvpe_dwconv_bias_silu_nhwc: K*K*C too large for shared memory");
  static thread_local uint64_t attr_set = 0;
  if (first_use_on_device(attr_set)) {
#define CCVPE_DW_ATTR(KK, SS) \
  cudaFuncSetAttribute(dwconv_bias_silu_kernel<KK, SS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)
    CCVPE_DW_ATTR(3, 1); CCVPE_DW_ATTR(3, 2); CCVPE_DW_ATTR(5, 1); CCVPE_DW_ATTR(5, 2);
#undef CCVPE_DW_ATTR
  }
  cudaStream_t st = (cudaStream_t)stream;
#define CCVPE_DW(KK, SS)                                                                                              \
  dwconv_bias_silu_kernel<KK, SS><<<grid, 256, sm, st>>>((const __nv_bfloat16*)x, x_sb, x_sh, x_sw,                   \
                                                         (const __nv_bfloat16*)w, (const __nv_bfloat16*)bias,         \
                                                         (__nv_bfloat16*)y, Ho, Wo, C, CG, (int)spb, reinterpret_cast<long long*>(chan_sum))
  if (K == 3 && S == 1) CCVPE_DW(3, 1);
  else if (K == 3 && S == 2) CCVPE_DW(3, 2);
  else if (K == 5 && S == 1) CCVPE_DW(5, 1);
  else CCVPE_DW(5, 2);
#undef CCVPE_DW
  CCVPE_LAUNCH_CHECK("dwconv_bias_silu_kernel");
  return CCVPE_OK;
}

extern "C" int ccvpe_dwconv_plan(int B, int C, int Hp, int Wp, int K, int S) {
  ccvpe::DwTileParams tp;
  return ccvpe::dw_select(B, C, Hp, Wp, K, S, &tp);
}
