// Sequential location filter: one Bayes-filter step per frame that fuses each heatmap with the motion-propagated belief of
// the previous frame (semantics in include/ccvpe_b200.h, ccvpe_track_step).
//
// Three launches per step, all on the caller's stream, no host synchronisation:
//   1. track_warp_hblur_kernel -- one CTA per (row, track): warps the old belief into the row (float64 source coordinates
//      with explicit _rn intrinsics, as affine.cu), stages it in shared memory and writes its horizontal Gaussian blur to
//      the scratch plane;
//   2. track_vblur_update_kernel -- one CTA per 32-column x 64-row tile: stages the tile's rows of the scratch plane with
//      an r-row halo above and below, blurs vertically, mixes in the uniform floor, multiplies by the heatmap in float64,
//      stores q (rounded to float32) over the belief and one float64 partial sum of q per CTA;
//   3. track_normalize_kernel -- every CTA of a track folds that track's partials in the same fixed order (so all of them
//      get the same Z bit for bit), CTA 0 writes evidence and reset, and each CTA scales its share of q by 1 / Z, or copies
//      the heatmap where Z is not a positive finite number.
// The blur weights are computed on the host (float64, rounded once to float32) and passed by value, so a captured step
// keeps its sigma; `motion` is read when the kernel runs, so a replay uses whatever the tensor holds.  Every sum is a
// fixed sequence or tree, so the output is a function of the inputs alone.
#include <cmath>

#include "common.cuh"

namespace ccvpe {
namespace {

constexpr int kTrackMaxRadius = 96;                // ceil(3 * 32)
constexpr float kTrackMaxSigma = 32.f;
constexpr int kTrackMaxDim = 4096;
constexpr int kTrackRowThreads = 256;              // launch 1: one row per CTA
constexpr int kTrackTileW = 32, kTrackTileH = 64;  // launch 2: output tile
constexpr int kTrackTileRowsMax = kTrackTileH + 2 * kTrackMaxRadius;
static_assert(kTrackTileH % 8 == 0, "launch 2 has 8 rows of threads");
constexpr int kTrackNormThreads = 256;
constexpr int kTrackNormPixelsPerCta = 16 * kTrackNormThreads;
constexpr int kTrackNormMaxCtas = 256;             // per track

struct TrackBlur {
  int r;                                           // radius: ceil(3 sigma), 0 for sigma = 0
  float w[kTrackMaxRadius + 1];                    // w[|d|], normalised over d in [-r, r]
};

// w[0] * s[0] + sum_{d=1..r} w[d] * (s[-d] + s[d]), accumulated in float32 in that order; s points at the output's tap in
// a shared-memory line whose r entries on either side are staged (zeros beyond the map's edge)
__device__ __forceinline__ float blur_at(const float* s, int stride, const float* w, int r) {
  float acc = w[0] * s[0];
  for (int d = 1; d <= r; ++d) acc = fmaf(w[d], s[-d * stride] + s[d * stride], acc);
  return acc;
}

// the blur weights into shared memory (a warp reads one broadcast word per tap)
__device__ __forceinline__ void stage_weights(float* w, const TrackBlur& g, int tid, int nthreads) {
  for (int d = tid; d <= g.r; d += nthreads) w[d] = g.w[d];
}

// Launch 1: belief[b] warped to the new grid (bilinear, zero padding, times |det|), then blurred along each row.
__global__ void __launch_bounds__(kTrackRowThreads)
track_warp_hblur_kernel(const float* __restrict__ belief, const double* __restrict__ motion, float* __restrict__ hb,
                        int H, int W, const TrackBlur g) {
  __shared__ float row[kTrackMaxDim + 2 * kTrackMaxRadius];   // the warped row with r zeros on either side
  __shared__ float w[kTrackMaxRadius + 1];
  const int i = blockIdx.x, b = blockIdx.y, r = g.r;
  stage_weights(w, g, threadIdx.x, kTrackRowThreads);
  for (int k = threadIdx.x; k < r; k += kTrackRowThreads) row[k] = row[r + W + k] = 0.f;
  const int64_t plane = (int64_t)H * W;
  const float* src = belief + b * plane;
  const double* a = motion + 6 * (int64_t)b;
  const double a0 = __ldg(a + 0), a1 = __ldg(a + 1), a2 = __ldg(a + 2), a3 = __ldg(a + 3), a4 = __ldg(a + 4),
               a5 = __ldg(a + 5);
  const float jac = (float)fabs(__dsub_rn(__dmul_rn(a0, a4), __dmul_rn(a1, a3)));
  const double yc = __dadd_rn((double)i, 0.5);
  const double a1y = __dmul_rn(a1, yc), a4y = __dmul_rn(a4, yc);
  for (int j = threadIdx.x; j < W; j += kTrackRowThreads) {
    const double xc = __dadd_rn((double)j, 0.5);
    const double u = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(a0, xc), a1y), a2), 0.5);
    const double v = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(a3, xc), a4y), a5), 0.5);
    const double uf = floor(u), vf = floor(v);
    float val = 0.f;
    // written as "some tap is inside" so that a NaN, infinite or huge coordinate gives 0 before any conversion to int
    if (uf >= -1.0 && uf <= (double)(W - 1) && vf >= -1.0 && vf <= (double)(H - 1)) {
      const double dx = __dsub_rn(u, uf), dy = __dsub_rn(v, vf);
      const float wx1 = (float)dx, wx0 = (float)__dsub_rn(1.0, dx), wy1 = (float)dy, wy0 = (float)__dsub_rn(1.0, dy);
      const int x0 = (int)uf, y0 = (int)vf, x1 = x0 + 1, y1 = y0 + 1;
      const bool cx0 = x0 >= 0, cx1 = x1 < W, cy0 = y0 >= 0, cy1 = y1 < H;
      float r0 = 0.f, r1 = 0.f;
      if (cy0) {
        const float* p = src + (int64_t)y0 * W;
        if (cx0) r0 = wx0 * __ldg(p + x0);
        if (cx1) r0 = fmaf(wx1, __ldg(p + x1), r0);
      }
      if (cy1) {
        const float* p = src + (int64_t)y1 * W;
        if (cx0) r1 = wx0 * __ldg(p + x0);
        if (cx1) r1 = fmaf(wx1, __ldg(p + x1), r1);
      }
      val = fmaf(wy0, r0, wy1 * r1) * jac;
    }
    row[r + j] = val;
  }
  __syncthreads();
  float* dst = hb + b * plane + (int64_t)i * W;
  for (int j = threadIdx.x; j < W; j += kTrackRowThreads) dst[j] = blur_at(row + r + j, 1, w, r);
}

// Launch 2: vertical blur of the scratch plane, the uniform mix and the product with the heatmap (float64); q rounded to
// float32 goes over the belief, the tile's float64 sum of q to partial[b][tile].
__global__ void __launch_bounds__(kTrackTileW * 8)
track_vblur_update_kernel(const float* __restrict__ hb, const float* __restrict__ heatmap, float* __restrict__ belief,
                          double* __restrict__ partial, int H, int W, const TrackBlur g, double keep, double floor_p) {
  constexpr int kRowsPerThread = kTrackTileH / 8;
  __shared__ float tile[kTrackTileRowsMax * kTrackTileW];             // rows [i0 - r, i0 + 64 + r), zeros off the map
  __shared__ float w[kTrackMaxRadius + 1];
  __shared__ double warp_sums[8];
  const int tx = threadIdx.x, ty = threadIdx.y, b = blockIdx.z, r = g.r;
  const int j = blockIdx.x * kTrackTileW + tx, i0 = blockIdx.y * kTrackTileH;
  const int64_t plane = (int64_t)H * W;
  // the heatmap values first, so that their loads overlap the staging below
  float h[kRowsPerThread];
#pragma unroll
  for (int k = 0; k < kRowsPerThread; ++k) {
    const int i = i0 + ty + 8 * k;
    h[k] = (j < W && i < H) ? __ldg(heatmap + b * plane + (int64_t)i * W + j) : 0.f;
  }
  stage_weights(w, g, ty * kTrackTileW + tx, kTrackTileW * 8);
  const int n_rows = kTrackTileH + 2 * r;
#pragma unroll 4
  for (int k = ty; k < n_rows; k += 8) {
    const int rr = i0 - r + k;
    tile[k * kTrackTileW + tx] = (j < W && rr >= 0 && rr < H) ? __ldg(hb + b * plane + (int64_t)rr * W + j) : 0.f;
  }
  __syncthreads();
  double sum = 0.0;
#pragma unroll
  for (int k = 0; k < kRowsPerThread; ++k) {
    const int i = i0 + ty + 8 * k;
    if (j < W && i < H) {
      const float p = blur_at(tile + (r + ty + 8 * k) * kTrackTileW + tx, kTrackTileW, w, r);
      const double prior = __dadd_rn(__dmul_rn(keep, (double)p), floor_p);
      const double q = __dmul_rn(prior, (double)h[k]);
      belief[b * plane + (int64_t)i * W + j] = (float)q;
      sum = __dadd_rn(sum, q);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
  if (tx == 0) warp_sums[ty] = sum;
  __syncthreads();
  if (tx == 0 && ty == 0) {
    double s = warp_sums[0];
    for (int w = 1; w < 8; ++w) s = __dadd_rn(s, warp_sums[w]);
    partial[(int64_t)b * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x] = s;
  }
}

// Launch 3: Z = the fixed-order fold of the track's partials; belief = q / Z, or the heatmap where Z is not in (0, inf).
__global__ void __launch_bounds__(kTrackNormThreads)
track_normalize_kernel(float* __restrict__ belief, const float* __restrict__ heatmap, const double* __restrict__ partial,
                       int n_partial, int64_t plane, double* __restrict__ evidence, uint8_t* __restrict__ reset) {
  __shared__ double warp_sums[kTrackNormThreads / 32];
  const int b = blockIdx.y, t = threadIdx.x;
  const double* pb = partial + (int64_t)b * n_partial;
  double s = 0.0;
  for (int k = t; k < n_partial; k += kTrackNormThreads) s = __dadd_rn(s, __ldg(pb + k));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
  if ((t & 31) == 0) warp_sums[t >> 5] = s;
  __syncthreads();
  double z = warp_sums[0];
  for (int w = 1; w < kTrackNormThreads / 32; ++w) z = __dadd_rn(z, warp_sums[w]);
  const bool ok = z > 0.0 && z <= 1.7976931348623157e308;  // false for NaN and +inf
  if (blockIdx.x == 0 && t == 0) {
    evidence[b] = z;
    reset[b] = ok ? 0 : 1;
  }
  float* q = belief + b * plane;
  const float* src = ok ? q : heatmap + b * plane;
  const double inv = 1.0 / z;
  const int64_t stride = (int64_t)gridDim.x * kTrackNormThreads;
  // 4 loads in flight per thread before the stores
  for (int64_t p0 = (int64_t)blockIdx.x * kTrackNormThreads + t; p0 < plane; p0 += 4 * stride) {
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = p0 + k * stride < plane ? src[p0 + k * stride] : 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (p0 + k * stride < plane) q[p0 + k * stride] = ok ? (float)__dmul_rn((double)v[k], inv) : v[k];
  }
}

struct TrackGeom {
  int tiles_x, tiles_y, n_partial, norm_ctas;
  int64_t partial_bytes, bytes;
};

TrackGeom track_geom(int B, int H, int W) {
  TrackGeom g;
  g.tiles_x = (W + kTrackTileW - 1) / kTrackTileW;
  g.tiles_y = (H + kTrackTileH - 1) / kTrackTileH;
  g.n_partial = g.tiles_x * g.tiles_y;
  const int64_t plane = (int64_t)H * W;
  g.norm_ctas = (int)std::min<int64_t>((plane + kTrackNormPixelsPerCta - 1) / kTrackNormPixelsPerCta, kTrackNormMaxCtas);
  g.partial_bytes = ((int64_t)B * g.n_partial * 8 + 255) / 256 * 256;
  g.bytes = g.partial_bytes + (int64_t)B * plane * 4;
  return g;
}

bool track_shape_ok(int B, int H, int W) {
  return B >= 1 && B <= 65535 && H >= 1 && H <= kTrackMaxDim && W >= 1 && W <= kTrackMaxDim;
}

}  // namespace
}  // namespace ccvpe

extern "C" int64_t ccvpe_track_scratch_bytes(int B, int H, int W) {
  if (!ccvpe::track_shape_ok(B, H, W)) return -1;
  return ccvpe::track_geom(B, H, W).bytes;
}

extern "C" int ccvpe_track_step(float* belief, const float* heatmap, const double* motion, int B, int H, int W,
                                float sigma, float epsilon, double* evidence, uint8_t* reset, void* scratch,
                                void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(belief && heatmap && motion && evidence && reset && scratch, "ccvpe_track_step: null pointer");
  CCVPE_REQUIRE(track_shape_ok(B, H, W), "ccvpe_track_step: bad shape B=%d H=%d W=%d (1 <= B <= 65535, 1 <= H, W <= %d)",
                B, H, W, kTrackMaxDim);
  CCVPE_REQUIRE(sigma >= 0.f && sigma <= kTrackMaxSigma, "ccvpe_track_step: sigma=%g outside [0, %g] pixels",
                (double)sigma, (double)kTrackMaxSigma);
  CCVPE_REQUIRE(epsilon >= 0.f && epsilon <= 1.f, "ccvpe_track_step: epsilon=%g outside [0, 1]", (double)epsilon);
  CCVPE_REQUIRE((((uintptr_t)belief | (uintptr_t)heatmap) & 3u) == 0 &&
                (((uintptr_t)motion | (uintptr_t)evidence | (uintptr_t)scratch) & 7u) == 0,
                "ccvpe_track_step: misaligned pointer");
  const int64_t bytes = (int64_t)B * H * W * 4;
  const uintptr_t bl = (uintptr_t)belief, hm = (uintptr_t)heatmap;
  CCVPE_REQUIRE(bl + bytes <= hm || hm + bytes <= bl, "ccvpe_track_step: heatmap overlaps belief");
  const TrackGeom geo = track_geom(B, H, W);
  TrackBlur g;
  g.r = (int)std::ceil(3.0 * (double)sigma);
  if (g.r == 0) {
    g.w[0] = 1.f;
  } else {
    double w[kTrackMaxRadius + 1], s = 0.0;
    const double s2 = 2.0 * (double)sigma * (double)sigma;
    for (int d = 0; d <= g.r; ++d) {
      w[d] = std::exp(-(double)d * d / s2);
      s += d ? 2.0 * w[d] : w[d];
    }
    for (int d = 0; d <= g.r; ++d) g.w[d] = (float)(w[d] / s);
  }
  const double keep = 1.0 - (double)epsilon, floor_p = (double)epsilon / ((double)H * W);
  double* partial = (double*)scratch;
  float* hb = (float*)((char*)scratch + geo.partial_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  track_warp_hblur_kernel<<<dim3(H, B), kTrackRowThreads, 0, st>>>(belief, motion, hb, H, W, g);
  CCVPE_LAUNCH_CHECK("track_warp_hblur_kernel");
  track_vblur_update_kernel<<<dim3(geo.tiles_x, geo.tiles_y, B), dim3(kTrackTileW, 8), 0, st>>>(
      hb, heatmap, belief, partial, H, W, g, keep, floor_p);
  CCVPE_LAUNCH_CHECK("track_vblur_update_kernel");
  track_normalize_kernel<<<dim3(geo.norm_ctas, B), kTrackNormThreads, 0, st>>>(belief, heatmap, partial, geo.n_partial,
                                                                              (int64_t)H * W, evidence, reset);
  CCVPE_LAUNCH_CHECK("track_normalize_kernel");
  return CCVPE_OK;
}
