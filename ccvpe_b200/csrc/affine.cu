// f4 -- geometric augmentation of decoded uint8 images on the device: Pillow's 8-bit BILINEAR affine transform
// (Image.transform(size, AFFINE, a, BILINEAR, fillcolor); Image.rotate(angle, BILINEAR, center, translate) builds such an
// `a`), bit-identical to Pillow (Geometry.c: affine_transform + bilinear_filter32RGB).  Per output pixel (x, y) of the
// untransformed-size result and per image matrix a[0..5] (output -> input coordinates):
//     xi = ((a0 * (x + 0.5)) + (a1 * (y + 0.5))) + a2,  yi = ((a3 * (x + 0.5)) + (a4 * (y + 0.5))) + a5
//     outside [0, W) x [0, H): the fill colour; otherwise, with xi -= 0.5, yi -= 0.5, (xf, yf) their floors, (dx, dy) the
//     fractions and x0, x1, y0 clamped into the image:
//     v1 = s[y0][x0] + (s[y0][x1] - s[y0][x0]) * dx;   v2 = row yf + 1 likewise if it is inside the image, else v1
//     out = (uint8) trunc(v1 + (v2 - v1) * dy)                                                     (per channel, in double)
// Every double operation is an explicit _rn intrinsic: nvcc contracts a * b + c into an FMA by default (doubles too),
// and Pillow's x86-64 build does not.
// One thread per output pixel, all three channels; a CTA owns a 32 x 8 tile of one image and gathers its source taps
// through L1 (neighbouring pixels share most of their taps).  The matrices are read from device memory and nothing is
// copied from the host, so a CUDA graph can be replayed with the matrices rewritten in place.
#include "common.cuh"

namespace ccvpe {

constexpr int kAffineTileW = 32, kAffineTileH = 8;

// Pillow's BILINEAR(v, a, b, d): v = a + (b - a) * d, in double, not fused
__device__ __forceinline__ double pil_lerp(double a, double b, double d) { return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), d)); }

template <bool NHWC>
__global__ void __launch_bounds__(kAffineTileW * kAffineTileH)
affine_u8_kernel(const uint8_t* __restrict__ src, const double* __restrict__ mat, uint8_t* __restrict__ dst, int H, int W,
                 int out_h, int out_w, int left, int top, uint32_t fill) {
  const int x = blockIdx.x * kAffineTileW + threadIdx.x, y = blockIdx.y * kAffineTileH + threadIdx.y;
  if (x >= out_w || y >= out_h) return;
  const int b = blockIdx.z;
  const double* a = mat + 6 * (int64_t)b;
  const double xc = __dadd_rn((double)(x + left), 0.5), yc = __dadd_rn((double)(y + top), 0.5);
  double xi = __dadd_rn(__dadd_rn(__dmul_rn(__ldg(a + 0), xc), __dmul_rn(__ldg(a + 1), yc)), __ldg(a + 2));
  double yi = __dadd_rn(__dadd_rn(__dmul_rn(__ldg(a + 3), xc), __dmul_rn(__ldg(a + 4), yc)), __ldg(a + 5));
  uint32_t v[3] = {fill & 255u, (fill >> 8) & 255u, (fill >> 16) & 255u};
  // written as "inside" so that a NaN coordinate takes the fill colour
  if (xi >= 0.0 && xi < (double)W && yi >= 0.0 && yi < (double)H) {
    xi = __dsub_rn(xi, 0.5);
    yi = __dsub_rn(yi, 0.5);
    const double xf = floor(xi), yf = floor(yi);
    const double dx = __dsub_rn(xi, xf), dy = __dsub_rn(yi, yf);
    const int ix = (int)xf, iy = (int)yf;  // in [-1, W - 1] and [-1, H - 1]
    const int x0 = max(ix, 0), x1 = min(ix + 1, W - 1), y0 = max(iy, 0), y1 = iy + 1;
    const bool row1 = y1 < H;
    // channel c of source pixel (row, col) is p[(row * W + col) * cs + c * ps]
    const int64_t cs = NHWC ? 3 : 1, ps = NHWC ? 1 : (int64_t)H * W;
    const uint8_t* p = src + (int64_t)b * 3 * H * W;
    const int64_t o00 = ((int64_t)y0 * W + x0) * cs, o01 = ((int64_t)y0 * W + x1) * cs;
    const int64_t o10 = ((int64_t)(row1 ? y1 : y0) * W + x0) * cs, o11 = ((int64_t)(row1 ? y1 : y0) * W + x1) * cs;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const uint8_t* q = p + c * ps;
      const double v1 = pil_lerp((double)__ldg(q + o00), (double)__ldg(q + o01), dx);
      const double v2 = row1 ? pil_lerp((double)__ldg(q + o10), (double)__ldg(q + o11), dx) : v1;
      v[c] = (uint32_t)__double2int_rz(pil_lerp(v1, v2, dy));  // in [0, 255]
    }
  }
  const int64_t plane = (int64_t)out_h * out_w;
  uint8_t* q = dst + (int64_t)b * 3 * plane + (int64_t)y * out_w + x;
  q[0] = (uint8_t)v[0];
  q[plane] = (uint8_t)v[1];
  q[2 * plane] = (uint8_t)v[2];
}

}  // namespace ccvpe

extern "C" int ccvpe_affine_u8(const uint8_t* src, int nhwc, int B, int H, int W, const double* matrices, int out_h,
                               int out_w, int left, int top, const uint8_t* fill_host, uint8_t* dst, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(src && matrices && fill_host && dst, "ccvpe_affine_u8: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && out_h > 0 && out_w > 0, "ccvpe_affine_u8: bad shape B=%d H=%d W=%d -> %dx%d",
                B, H, W, out_h, out_w);
  CCVPE_REQUIRE(left >= 0 && top >= 0 && (int64_t)left + out_w <= INT32_MAX && (int64_t)top + out_h <= INT32_MAX,
                "ccvpe_affine_u8: bad offset (left=%d, top=%d) for a %dx%d output", left, top, out_h, out_w);
  CCVPE_REQUIRE(B <= 65535, "ccvpe_affine_u8: B=%d exceeds 65535 images per call", B);
  const int64_t tiles_y = ((int64_t)out_h + kAffineTileH - 1) / kAffineTileH;
  CCVPE_REQUIRE(tiles_y <= 65535, "ccvpe_affine_u8: output %dx%d too large", out_h, out_w);
  const uint32_t fill = fill_host[0] | (uint32_t)fill_host[1] << 8 | (uint32_t)fill_host[2] << 16;
  const dim3 grid((unsigned)((out_w + kAffineTileW - 1) / kAffineTileW), (unsigned)tiles_y, (unsigned)B);
  const dim3 block(kAffineTileW, kAffineTileH);
  cudaStream_t st = (cudaStream_t)stream;
  if (nhwc)
    affine_u8_kernel<true><<<grid, block, 0, st>>>(src, matrices, dst, H, W, out_h, out_w, left, top, fill);
  else
    affine_u8_kernel<false><<<grid, block, 0, st>>>(src, matrices, dst, H, W, out_h, out_w, left, top, fill);
  CCVPE_LAUNCH_CHECK("affine_u8_kernel");
  return CCVPE_OK;
}
