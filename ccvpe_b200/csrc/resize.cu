// f4 -- the reference's transforms.Resize(size) on PIL images (train_VIGOR.py:55-70; Image.resize(.., BILINEAR)) on the
// device, bit-identical to Pillow's 8-bit resampler (Resample.c: precompute_coeffs, normalize_coeffs_8bpc,
// ImagingResampleHorizontal_8bpc / Vertical_8bpc).  Per axis, output index o reads the source window [xmin, xmin + n) with
// integer weights k (2^22 fixed point) computed in double precision; the horizontal pass runs first into a uint8
// intermediate, then the vertical pass over it:
//     inter[y, o] = clip8((2^21 + sum_x src[y, xmin_o + x] * kh_o[x]) >> 22)
//     dst[o', o]  = clip8((2^21 + sum_y inter[ymin_o' + y, o] * kv_o'[y]) >> 22)
// One kernel: a CTA owns a TH x TW output tile (all three channels) of a few images, computes the tile's coefficients
// into shared memory once, and for each image streams the tile's source window through shared memory in row chunks
// (16-byte cp.async copies), runs the horizontal pass into a shared uint8 intermediate and the vertical pass from it,
// so HBM sees the window once and the output once.  The library
// never copies coefficient tables from the host: the kernel needs no workspace and is capturable in a CUDA graph.
#include <math.h>

#include "common.cuh"

namespace ccvpe {

constexpr int kResizeThreads = 256;
constexpr int kResizeSmemBudget = 64 * 1024;  // three to four CTAs per SM at the VIGOR sizes
constexpr int kPrecisionBits = 22;            // Pillow's PRECISION_BITS for 8 bits per channel

__device__ __forceinline__ uint8_t clip8(int s) {
  return s >= (1 << kPrecisionBits << 8) ? 255 : (s <= 0 ? 0 : (uint8_t)(s >> kPrecisionBits));
}

// Pillow's bilinear filter at source index x (x + xmin in precompute_coeffs) around `center`; ss = 1 / filterscale.
__device__ __forceinline__ double tri_weight(int x, double center, double ss) {
  const double t = fabs(__dmul_rn(__dadd_rn(__dsub_rn((double)x, center), 0.5), ss));
  return t < 1.0 ? __dsub_rn(1.0, t) : 0.0;
}

// Pillow's precompute_coeffs + normalize_coeffs_8bpc.  Every double operation is an explicit _rn intrinsic: nvcc
// contracts a * b + c into an FMA by default (doubles too), and Pillow's x86-64 build does not.
struct PilAxis {
  int in;
  double scale, fs, ss;  // in / out, filterscale = max(scale, 1) (support = 1.0 * filterscale), 1 / filterscale
};
__device__ inline PilAxis pil_axis(int in, int out) {
  PilAxis a;
  a.in = in;
  a.scale = __ddiv_rn((double)in, (double)out);
  a.fs = a.scale < 1.0 ? 1.0 : a.scale;
  a.ss = __ddiv_rn(1.0, a.fs);
  return a;
}
__device__ inline double pil_center(const PilAxis& a, int o) { return __dmul_rn(__dadd_rn((double)o, 0.5), a.scale); }
// window [xmin, xmin + n) of output o and ww, the sequential (Pillow-order) sum of its unnormalised weights
__device__ __forceinline__ void pil_window(const PilAxis& a, int o, int* xmin_out, int* n_out, double* ww_out) {
  const double center = pil_center(a, o);
  int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, a.fs), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, a.fs), 0.5));
  if (xmax > a.in) xmax = a.in;
  double ww = 0.0;
  for (int x = xmin; x < xmax; ++x) ww = __dadd_rn(ww, tri_weight(x, center, a.ss));
  *xmin_out = xmin;
  *n_out = xmax - xmin;
  *ww_out = ww;
}
// 2^22 fixed-point weight of source index x (inside the window) of output o
__device__ inline int32_t pil_weight(const PilAxis& a, int o, int x, double ww) {
  double w = tri_weight(x, pil_center(a, o), a.ss);
  if (ww != 0.0) w = __ddiv_rn(w, ww);
  return __double2int_rz(__dadd_rn(0.5, __dmul_rn(w, (double)(1 << kPrecisionBits))));  // w >= 0
}

// Tile geometry shared by the launcher (sizing) and the kernel (carving shared memory).
struct ResizeTile {
  int th, tw;          // output tile
  int kh, kv;          // Pillow's ksize per axis (upper bound of n)
  int rows_max;        // bound of the source rows one tile reads (intermediate height)
  int cols_max;        // bound of the source columns one tile reads
  int rc;              // source rows staged per chunk
  int pitch;           // bytes per staged source segment (one NHWC row, or one channel of an NCHW row), 16-aligned
  int nb;              // images per CTA (the tile's coefficients are computed once for all of them)
  int smem;            // dynamic shared memory bytes
};

// 64-bit: the launcher sizes candidate tiles whose tables are far larger than shared memory before it refuses them
__host__ __device__ inline int64_t coef_bytes(const ResizeTile& t) {
  return 8 * ((int64_t)t.tw + t.th) + 4 * (2 * (int64_t)t.tw + 2 * t.th + (int64_t)t.kh * t.tw + (int64_t)t.kv * t.th);
}
__host__ __device__ inline int64_t stage_offset(const ResizeTile& t) {
  return (coef_bytes(t) + 3 * (int64_t)t.rows_max * t.tw + 15) & ~(int64_t)15;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gmem_src)
               : "memory");
}

template <bool NHWC>
__global__ void __launch_bounds__(kResizeThreads, 4)
resize_u8_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int B, int H, int W, int out_h, int out_w,
                 ResizeTile tl) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int TW = tl.tw, TH = tl.th;
  double* hww = reinterpret_cast<double*>(smem);  // [TW] weight sum of each output column
  double* vww = hww + TW;                         // [TH] ... of each output row
  int* hx = reinterpret_cast<int*>(vww + TH);     // [TW] first source column of each output column
  int* hn = hx + TW;                              // [TW] its tap count
  int* vy = hn + TW;                              // [TH] first source row of each output row
  int* vn = vy + TH;
  int32_t* hk = vn + TH;                          // [kh][TW] tap-major: lanes of a warp read consecutive words
  int32_t* vk = hk + tl.kh * TW;                  // [kv][TH]
  uint8_t* inter = smem + coef_bytes(tl);         // [3][rows_max][TW]
  uint8_t* stage = smem + stage_offset(tl);

  const int tid = threadIdx.x;
  const int ox0 = blockIdx.x * TW, oy0 = blockIdx.y * TH;
  const int tw = min(TW, out_w - ox0), th = min(TH, out_h - oy0);
  // coefficients: the windows and weight sums one thread per output, then the weights one thread per (output, tap)
  const PilAxis ah = pil_axis(W, out_w), av = pil_axis(H, out_h);
  for (int i = tid; i < tw + th; i += kResizeThreads) {
    if (i < tw)
      pil_window(ah, ox0 + i, hx + i, hn + i, hww + i);
    else
      pil_window(av, oy0 + i - tw, vy + i - tw, vn + i - tw, vww + i - tw);
  }
  __syncthreads();
  const int nh = tw * tl.kh;
  for (int i = tid; i < nh + th * tl.kv; i += kResizeThreads) {
    if (i < nh) {
      const int o = i / tl.kh, x = i - o * tl.kh;
      if (x < hn[o]) hk[x * TW + o] = pil_weight(ah, ox0 + o, hx[o] + x, hww[o]);
    } else {
      const int o = (i - nh) / tl.kv, x = i - nh - o * tl.kv;
      if (x < vn[o]) vk[x * TH + o] = pil_weight(av, oy0 + o, vy[o] + x, vww[o]);
    }
  }
  __syncthreads();
  // the windows are monotone in the output index, so the tile's window runs from the first start to the last end
  const int sx0 = hx[0], ncols = hx[tw - 1] + hn[tw - 1] - sx0;
  const int sy0 = vy[0], nrows = vy[th - 1] + vn[th - 1] - sy0;
  constexpr int kSegs = NHWC ? 1 : 3;
  const int len = NHWC ? ncols * 3 : ncols;
  const int pv = tl.pitch >> 4;

  int b;
  // source segment s (row s / kSegs of the chunk, channel s % kSegs for NCHW) of image b in global memory, and where it
  // starts in its staged copy (the low 4 bits of its address; 32-bit arithmetic keeps them)
  auto seg_src = [&](int r0, int s) -> const uint8_t* {
    const int y = sy0 + r0 + s / kSegs;
    return NHWC ? src + (((int64_t)b * H + y) * W + sx0) * 3 : src + (((int64_t)b * 3 + s % kSegs) * H + y) * W + sx0;
  };
  auto seg_stage = [&](int r0, int s) -> const uint8_t* {
    const uint32_t y = sy0 + r0 + s / kSegs, ub = b, uH = H, uW = W, ux = sx0;
    const uint32_t off = NHWC ? ((ub * uH + y) * uW + ux) * 3u : ((ub * 3u + s % kSegs) * uH + y) * uW + ux;
    return stage + s * tl.pitch + (((uint32_t)reinterpret_cast<uintptr_t>(src) + off) & 15u);
  };
  // passes: thread (j, rg) owns output column j of the tile, for rows rg, rg + rstep, ... and all three channels
  const int j = tid % TW, rg = tid / TW, rstep = kResizeThreads / TW;
  const int b_end = min(B, (int)(blockIdx.z + 1) * tl.nb);

  for (b = blockIdx.z * tl.nb; b < b_end; ++b) {
    for (int r0 = 0; r0 < nrows; r0 += tl.rc) {
      const int rn = min(tl.rc, nrows - r0);
      // stage: segment s lands at stage + s * pitch + (its global address & 15), so every full 16-byte word is one
      // asynchronous copy
      for (int i = tid; i < rn * kSegs * pv; i += kResizeThreads) {
        const int s = i / pv, v = i - s * pv;
        const uint8_t* g = seg_src(r0, s);
        const int lo = v * 16 - (int)(reinterpret_cast<uintptr_t>(g) & 15);
        if (lo >= len) continue;
        uint8_t* d = stage + s * tl.pitch + v * 16;
        if (lo >= 0 && lo + 16 <= len) {
          cp_async16(d, g + lo);
        } else {  // the segment's first or last word: only its own bytes are read
          uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
          for (int q = 0; q < 16; ++q)
            if (lo + q >= 0 && lo + q < len) w[q >> 2] |= (uint32_t)__ldg(g + lo + q) << (8 * (q & 3));
          *reinterpret_cast<uint4*>(d) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      asm volatile("cp.async.wait_all;\n" ::: "memory");
      __syncthreads();
      // horizontal pass of the chunk's rows into the intermediate
      if (j < tw) {
        const int xo = hx[j] - sx0, n = hn[j];
        for (int r = rg; r < rn; r += rstep) {
          // channel c of tap t is p_c[t * ps]
          const uint8_t *p0, *p1, *p2;
          if (NHWC) {
            p0 = seg_stage(r0, r) + xo * 3;
            p1 = p0 + 1;
            p2 = p0 + 2;
          } else {
            p0 = seg_stage(r0, 3 * r) + xo;
            p1 = seg_stage(r0, 3 * r + 1) + xo;
            p2 = seg_stage(r0, 3 * r + 2) + xo;
          }
          constexpr int ps = NHWC ? 3 : 1;
          int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
          for (int t = 0; t < n; ++t) {
            const int k = hk[t * TW + j];
            a0 += (int)p0[t * ps] * k;
            a1 += (int)p1[t * ps] * k;
            a2 += (int)p2[t * ps] * k;
          }
          uint8_t* q = inter + (r0 + r) * TW + j;
          q[0] = clip8(a0);
          q[tl.rows_max * TW] = clip8(a1);
          q[2 * tl.rows_max * TW] = clip8(a2);
        }
      }
      __syncthreads();
    }

    // vertical pass from the intermediate to the NCHW output (the next image's staging writes only `stage`, and its
    // horizontal pass starts after a barrier)
    if (j < tw) {
      const int cs = tl.rows_max * TW;  // channel stride of the intermediate
      for (int r = rg; r < th; r += rstep) {
        const uint8_t* p = inter + (vy[r] - sy0) * TW + j;
        const int n = vn[r];
        int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
        for (int t = 0; t < n; ++t) {
          const int k = vk[t * TH + r];
          a0 += (int)p[t * TW] * k;
          a1 += (int)p[cs + t * TW] * k;
          a2 += (int)p[2 * cs + t * TW] * k;
        }
        const int64_t plane = (int64_t)out_h * out_w;
        uint8_t* q = dst + (int64_t)b * 3 * plane + (int64_t)(oy0 + r) * out_w + ox0 + j;
        q[0] = clip8(a0);
        q[plane] = clip8(a1);
        q[2 * plane] = clip8(a2);
      }
    }
  }
}

// Host side of Pillow's axis set-up: ksize = 2 * ceil(support) + 1, and a bound of the source span of T consecutive
// outputs: xmax(o + T - 1) - xmin(o) <= (T - 1) * scale + 2 * support + 1.
struct AxisSize {
  double scale, support;
  int ksize;
};
static AxisSize axis_size(int in, int out) {
  AxisSize a;
  a.scale = (double)in / out;
  a.support = a.scale < 1.0 ? 1.0 : a.scale;
  a.ksize = 2 * (int)ceil(a.support) + 1;  // <= 2^25 + 1 for in < 2^24
  return a;
}
static int axis_span(const AxisSize& a, int in, int T) {
  const double e = (T - 1) * a.scale + 2.0 * a.support;
  return e + 3.0 >= (double)in ? in : (int)e + 3;
}

// Largest tile (64 x 16, halved alternately down to 1 x 1) whose coefficient tables, weight sums and uint8
// intermediate (all source rows of the tile, three channels) leave room for at least 8 staged source rows (or the whole
// window; one row for a one-pixel tile) within the shared-memory budget.  smem = -1 when not even 1 x 1 fits.
static ResizeTile plan_tile(bool nhwc, int H, int W, int out_h, int out_w) {
  const AxisSize ah = axis_size(W, out_w), av = axis_size(H, out_h);
  ResizeTile t;
  t.tw = 64;
  t.th = 16;
  t.kh = ah.ksize;
  t.kv = av.ksize;
  t.nb = 1;
  for (;;) {
    t.cols_max = axis_span(ah, W, t.tw);
    t.rows_max = axis_span(av, H, t.th);
    const int64_t pitch = ((nhwc ? 3 * (int64_t)t.cols_max : t.cols_max) + 15 + 15) & ~(int64_t)15;
    const int64_t row_bytes = (nhwc ? 1 : 3) * pitch;
    const int64_t fixed = stage_offset(t);
    const int64_t room = fixed < kResizeSmemBudget ? (kResizeSmemBudget - fixed) / row_bytes : 0;
    const int64_t need = (t.tw == 1 && t.th == 1) ? 1 : (t.rows_max < 8 ? t.rows_max : 8);
    if (room >= need) {
      t.pitch = (int)pitch;  // room >= 1: one staged row fits the budget
      t.rc = (int)(room < t.rows_max ? room : t.rows_max);
      t.smem = (int)(fixed + t.rc * row_bytes);
      return t;
    }
    if (t.th > 1 && (4 * t.th >= t.tw || t.tw == 1))
      t.th >>= 1;
    else if (t.tw > 1)
      t.tw >>= 1;
    else
      break;
  }
  t.smem = -1;
  return t;
}

}  // namespace ccvpe

extern "C" int ccvpe_resize_u8(const uint8_t* src, int nhwc, int B, int H, int W, int out_h, int out_w, uint8_t* dst,
                               void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(src && dst, "ccvpe_resize_u8: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && out_h > 0 && out_w > 0, "ccvpe_resize_u8: bad shape B=%d H=%d W=%d -> %dx%d",
                B, H, W, out_h, out_w);
  CCVPE_REQUIRE(H < (1 << 24) && W < (1 << 24), "ccvpe_resize_u8: H=%d W=%d: sizes must be below 2^24", H, W);
  CCVPE_REQUIRE(B <= 65535, "ccvpe_resize_u8: B=%d exceeds 65535 images per call", B);
  ResizeTile tl = plan_tile(nhwc != 0, H, W, out_h, out_w);
  CCVPE_REQUIRE(tl.smem > 0, "ccvpe_resize_u8: %dx%d -> %dx%d: downscale too large: one output pixel's coefficient tables "
                "(%d x %d taps) and its uint8 intermediate column do not fit in shared memory", H, W, out_h, out_w,
                tl.kv, tl.kh);
  const int64_t tiles_x = (out_w + tl.tw - 1) / tl.tw, tiles_y = (out_h + tl.th - 1) / tl.th;
  CCVPE_REQUIRE(tiles_y <= 65535 && tiles_x <= INT32_MAX, "ccvpe_resize_u8: output %dx%d too large", out_h, out_w);
  // several images per CTA amortise the tile's coefficients, while leaving ~16 CTAs per SM to spread over the GPU
  const int64_t want = 16LL * sm_count(), tiles = tiles_x * tiles_y;
  tl.nb = tiles * B > want ? (int)((tiles * B) / want) : 1;
  if (tl.nb > B) tl.nb = B;
  const dim3 grid((unsigned)tiles_x, (unsigned)tiles_y, (unsigned)((B + tl.nb - 1) / tl.nb));
  cudaStream_t st = (cudaStream_t)stream;
  static thread_local uint64_t attr_set = 0;
  if (first_use_on_device(attr_set)) {
    cudaError_t e = cudaFuncSetAttribute(resize_u8_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kResizeSmemBudget);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(resize_u8_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kResizeSmemBudget);
    if (e != cudaSuccess) {
      attr_set = 0;
      return fail(CCVPE_ERR_CUDA, "cudaFuncSetAttribute(resize_u8): %s", cudaGetErrorString(e));
    }
  }
  if (nhwc)
    resize_u8_kernel<true><<<grid, kResizeThreads, tl.smem, st>>>(src, dst, B, H, W, out_h, out_w, tl);
  else
    resize_u8_kernel<false><<<grid, kResizeThreads, tl.smem, st>>>(src, dst, B, H, W, out_h, out_w, tl);
  CCVPE_LAUNCH_CHECK("resize_u8_kernel");
  return CCVPE_OK;
}
