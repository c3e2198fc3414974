// f4 -- the scripts' input pipeline after image decoding, on the GPU (SURVEY section 8(f)-4):
//   transforms.ToTensor + Normalize(mean, std) (reference train_VIGOR.py:55-70), the random panorama roll
//   (torch.roll(grd, shift, dims=2), datasets.py:118) and the limited-FoV crop (grd[:, :, :, :int(W*FoV/360)],
//   train_VIGOR.py:272-273) in one pass over the uint8 image:
//       dst[b, c, h, w] = (src[b, c, h, (w - shift_b) mod W] / 255 - mean[c]) / std[c]            w < crop_w
// The host ships 1 byte per sample instead of 4 (the fp32 images were what bounded 8-GPU end-to-end throughput).  The
// arithmetic is the reference's, operation for operation (IEEE fp32 divide, subtract, divide), so the result is
// bit-identical to torchvision's transforms on the same uint8 pixels.  The Resize before it is resize.cu.
#include "common.cuh"

namespace ccvpe {

template <bool NHWC>
__global__ void __launch_bounds__(256)
ingest_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, int H, int W, int crop_w,
                 const int32_t* __restrict__ shift, float m0, float m1, float m2, float s0, float s1, float s2,
                 int64_t total4) {
  const int w4s = (crop_w + 3) >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int w0 = (int)(i % w4s) * 4;
    int64_t r = i / w4s;
    const int h = (int)(r % H);
    r /= H;
    const int c = (int)(r % 3);
    const int b = (int)(r / 3);
    const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2);
    const float sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
    int sh = shift ? shift[b] % W : 0;
    if (sh < 0) sh += W;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int ws = w0 + j - sh;                       // torch.roll: out[w] = in[(w - shift) mod W]
      if (ws < 0) ws += W;
      if (ws >= W) ws -= W;
      const int64_t si = NHWC ? (((int64_t)b * H + h) * W + ws) * 3 + c : (((int64_t)b * 3 + c) * H + h) * W + ws;
      const float x = (w0 + j < crop_w) ? (float)__ldg(src + si) : 0.f;
      v[j] = __fdiv_rn(__fsub_rn(__fdiv_rn(x, 255.f), mean), sd);
    }
    float* o = dst + (((int64_t)b * 3 + c) * H + h) * crop_w + w0;
    if (w0 + 4 <= crop_w && (crop_w & 3) == 0) {
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
      for (int j = 0; j < 4 && w0 + j < crop_w; ++j) o[j] = v[j];
    }
  }
}

}  // namespace ccvpe

extern "C" int ccvpe_ingest_u8(const uint8_t* src, int nhwc, int B, int H, int W, int crop_w, const int32_t* shift,
                               const float* mean_host, const float* std_host, float* dst, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(src && dst && mean_host && std_host, "ccvpe_ingest_u8: null pointer");
  CCVPE_REQUIRE(B > 0 && H > 0 && W > 0 && crop_w > 0 && crop_w <= W, "ccvpe_ingest_u8: bad shape B=%d H=%d W=%d crop_w=%d", B,
                H, W, crop_w);
  CCVPE_REQUIRE(aligned16(dst), "ccvpe_ingest_u8: dst must be 16-byte aligned");
  const int64_t total4 = (int64_t)B * 3 * H * ((crop_w + 3) / 4);
  int64_t blocks = (total4 + 255) / 256;
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  cudaStream_t st = (cudaStream_t)stream;
  if (nhwc)
    ingest_u8_kernel<true><<<(int)blocks, 256, 0, st>>>(src, dst, H, W, crop_w, shift, mean_host[0], mean_host[1], mean_host[2],
                                                        std_host[0], std_host[1], std_host[2], total4);
  else
    ingest_u8_kernel<false><<<(int)blocks, 256, 0, st>>>(src, dst, H, W, crop_w, shift, mean_host[0], mean_host[1], mean_host[2],
                                                         std_host[0], std_host[1], std_host[2], total4);
  CCVPE_LAUNCH_CHECK("ingest_u8_kernel");
  return CCVPE_OK;
}
