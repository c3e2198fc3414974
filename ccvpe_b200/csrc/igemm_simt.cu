// CUDA-core backend of the generic implicit GEMM (a3 cell descriptors, a8 transposed convs, a9 3x3 convs).
// fp32 FMA accumulation in registers, operands staged through shared memory; this is the exact-fp32 parity path
// (the tcgen05 backend in igemm_tcgen05.cu is the bf16 throughput path).
//
// Tile: 128 output pixels x 64 output channels x 16 input channels per step, 256 threads, 8x4 outputs per thread.
// The K loop walks taps x {source 0, source 1} x channel chunks, so torch.cat([x, skip]) is never materialised.
#include <cstdlib>

#include "common.cuh"

namespace ccvpe {

constexpr int SBM = 128, SBN = 64, SBK = 16, STHREADS = 256;

struct IgemmArgs {
  ccvpe_igemm_desc d;
  int M;      // B * Hout * Wout
  int ktot;   // c0 + c1
  int chunks0, chunks1;
};

template <typename T>
__global__ void __launch_bounds__(STHREADS) igemm_simt_kernel(const IgemmArgs args) {
  const ccvpe_igemm_desc& d = args.d;
  __shared__ __align__(16) float As[SBK][SBM + 4];
  __shared__ __align__(16) float Bs[SBK][SBN];

  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;
  const int m0 = blockIdx.x * SBM, n0 = blockIdx.y * SBN;
  const int HWo = d.Hout * d.Wout;

  // the two A rows this thread stages
  int a_b[2], a_h[2], a_w[2];
  bool a_ok[2];
  const int a_q = (t & 3) * 4;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    int m = m0 + (t >> 2) + j * 64;
    a_ok[j] = m < args.M;
    int mm = a_ok[j] ? m : 0;
    a_b[j] = mm / HWo;
    int r = mm - a_b[j] * HWo;
    a_h[j] = (r / d.Wout) * d.stride - d.pad;
    a_w[j] = (r % d.Wout) * d.stride - d.pad;
  }
  const int b_k = t >> 4, b_n = (t & 15) * 4;
  const bool n_vec = (d.N % 4 == 0);

  const T* src0 = static_cast<const T*>(d.a0);
  const T* src1 = static_cast<const T*>(d.a1);
  const T* wkn = static_cast<const T*>(d.w_kn);

  const int steps_per_tap = args.chunks0 + args.chunks1;
  const int taps = d.kh * d.kw;
  const int total_steps = taps * steps_per_tap;

  float4 ra[2];
  float4 rb;

  auto fetch = [&](int step) {
    int tap = step / steps_per_tap;
    int within = step - tap * steps_per_tap;
    int ty_tap = tap / d.kw, tx_tap = tap - ty_tap * d.kw;
    const T* src;
    int csrc, ld, koff, kc;
    if (within < args.chunks0) {
      src = src0; csrc = d.c0; ld = d.ld0; koff = 0; kc = within * SBK;
    } else {
      src = src1; csrc = d.c1; ld = d.ld1; koff = d.c0; kc = (within - args.chunks0) * SBK;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      int hi = a_h[j] + ty_tap, wi = a_w[j] + tx_tap;
      bool ok = a_ok[j] && hi >= 0 && hi < d.Hin && wi >= 0 && wi < d.Win && (kc + a_q) < csrc;
      ra[j] = ok ? load4(src + (((int64_t)a_b[j] * d.Hin + hi) * d.Win + wi) * ld + kc + a_q)
                 : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    rb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kc + b_k < csrc) {
      const T* wrow = wkn + ((int64_t)tap * args.ktot + koff + kc + b_k) * d.N + n0 + b_n;
      if (n_vec) {
        if (n0 + b_n < d.N) rb = load4(wrow);
      } else {
        if (n0 + b_n + 0 < d.N) rb.x = to_float(wrow[0]);
        if (n0 + b_n + 1 < d.N) rb.y = to_float(wrow[1]);
        if (n0 + b_n + 2 < d.N) rb.z = to_float(wrow[2]);
        if (n0 + b_n + 3 < d.N) rb.w = to_float(wrow[3]);
      }
    }
  };
  auto stage = [&]() {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      int row = (t >> 2) + j * 64;
      As[a_q + 0][row] = ra[j].x;
      As[a_q + 1][row] = ra[j].y;
      As[a_q + 2][row] = ra[j].z;
      As[a_q + 3][row] = ra[j].w;
    }
    *reinterpret_cast<float4*>(&Bs[b_k][b_n]) = rb;
  };

  float acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[r][j] = 0.f;

  fetch(0);
  stage();
  __syncthreads();
  for (int step = 0; step < total_steps; ++step) {
    if (step + 1 < total_steps) fetch(step + 1);
#pragma unroll
    for (int k = 0; k < SBK; ++k) {
      float4 a_lo = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      float4 a_hi = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      float av[8] = {a_lo.x, a_lo.y, a_lo.z, a_lo.w, a_hi.x, a_hi.y, a_hi.z, a_hi.w};
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        acc[r][0] = fmaf(av[r], bv.x, acc[r][0]);
        acc[r][1] = fmaf(av[r], bv.y, acc[r][1]);
        acc[r][2] = fmaf(av[r], bv.z, acc[r][2]);
        acc[r][3] = fmaf(av[r], bv.w, acc[r][3]);
      }
    }
    __syncthreads();
    if (step + 1 < total_steps) {
      stage();
      __syncthreads();
    }
  }

  // epilogue
  const int nb = n0 + tx * 4;
  float bias4[4] = {0.f, 0.f, 0.f, 0.f}, r1w4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (nb + j < d.N) {
      if (d.bias) bias4[j] = d.bias[nb + j];
      if (d.row_r1) r1w4[j] = d.r1_w[nb + j];
    }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    int m = m0 + ty * 8 + r;
    if (m >= args.M) continue;
    float rs = d.row_scale ? d.row_scale[m] : 1.f;
    float r1 = d.row_r1 ? d.row_r1[m] : 0.f;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float y = d.row_scale ? acc[r][j] * rs : acc[r][j];
      if (d.row_r1) y = fmaf(r1, r1w4[j], y);
      y += bias4[j];
      if (d.relu) y = fmaxf(y, 0.f);
      v[j] = y;
    }
    if (d.out_mode == 2) {
      int b = m / HWo, hw = m - b * HWo;
      float* o = static_cast<float*>(d.out);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (nb + j < d.N) o[((int64_t)b * d.N + nb + j) * HWo + hw] = v[j];
      continue;
    }
    int64_t base;
    int col = nb;
    if (d.out_mode == 0) {
      base = (int64_t)m * d.ldo;
    } else {  // pixel shuffle of the k2 s2 transposed conv: n = (i*2 + j)*Cout + co
      int cout = d.N >> 2;
      int ij = nb / cout;
      col = nb - ij * cout;
      int b = m / HWo, r2 = m - b * HWo;
      int h = r2 / d.Wout, w = r2 - h * d.Wout;
      base = (((int64_t)b * 2 * d.Hout + 2 * h + (ij >> 1)) * (2 * d.Wout) + 2 * w + (ij & 1)) * d.ldo;
    }
    if (nb + 3 < d.N && n_vec && (d.ldo & 3) == 0) {
      if (d.out_dtype == CCVPE_F32)
        store4(static_cast<float*>(d.out) + base + col, make_float4(v[0], v[1], v[2], v[3]));
      else
        store4(static_cast<__nv_bfloat16*>(d.out) + base + col, make_float4(v[0], v[1], v[2], v[3]));
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (nb + j < d.N) {
          if (d.out_dtype == CCVPE_F32) static_cast<float*>(d.out)[base + col + j] = v[j];
          else static_cast<__nv_bfloat16*>(d.out)[base + col + j] = __float2bfloat16_rn(v[j]);
        }
    }
  }
}

int igemm_simt(const ccvpe_igemm_desc& d, cudaStream_t st) {
  if (!d.w_kn) return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_igemm(SIMT): w_kn is null");
  IgemmArgs args;
  args.d = d;
  args.M = d.B * d.Hout * d.Wout;
  args.ktot = d.c0 + d.c1;
  args.chunks0 = (d.c0 + SBK - 1) / SBK;
  args.chunks1 = (d.c1 + SBK - 1) / SBK;
  dim3 grid((args.M + SBM - 1) / SBM, (d.N + SBN - 1) / SBN);
  if (d.dtype == CCVPE_F32)
    igemm_simt_kernel<float><<<grid, STHREADS, 0, st>>>(args);
  else
    igemm_simt_kernel<__nv_bfloat16><<<grid, STHREADS, 0, st>>>(args);
  return check_launch("igemm_simt_kernel");
}

int igemm_tcgen05(const ccvpe_igemm_desc& d, cudaStream_t st, const TcOutPad* out_pad);  // igemm_tcgen05.cu
bool igemm_tcgen05_supported(const ccvpe_igemm_desc& d);
int conv_ring_tcgen05(const ccvpe_igemm_desc& d, cudaStream_t st);  // conv_ring_tcgen05.cu
bool conv_ring_supported(const ccvpe_igemm_desc& d);

}  // namespace ccvpe

extern "C" int ccvpe_igemm_plan(const ccvpe_igemm_desc* desc) {
  using namespace ccvpe;
  CCVPE_REQUIRE(desc != nullptr, "ccvpe_igemm_plan: null descriptor");
  const ccvpe_igemm_desc& d = *desc;
  int backend = d.backend;
  if (backend == CCVPE_BACKEND_AUTO)
    backend = (d.dtype == CCVPE_BF16 && d.w_nk && igemm_tcgen05_supported(d)) ? CCVPE_BACKEND_TCGEN05
                                                                               : CCVPE_BACKEND_SIMT;
  if (backend == CCVPE_BACKEND_SIMT) return 0;
  if (backend == CCVPE_BACKEND_TCGEN05) return conv_ring_supported(d) ? 2 : 1;
  return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_igemm_plan: unknown backend %d", d.backend);
}

extern "C" int ccvpe_igemm(const ccvpe_igemm_desc* desc, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(desc != nullptr, "ccvpe_igemm: null descriptor");
  const ccvpe_igemm_desc& d = *desc;
  CCVPE_REQUIRE(d.a0 && d.out, "ccvpe_igemm: null a0/out");
  CCVPE_REQUIRE(d.dtype == CCVPE_F32 || d.dtype == CCVPE_BF16, "ccvpe_igemm: bad dtype %d", d.dtype);
  CCVPE_REQUIRE(d.out_dtype == CCVPE_F32 || d.out_dtype == CCVPE_BF16, "ccvpe_igemm: bad out_dtype %d", d.out_dtype);
  CCVPE_REQUIRE(d.B > 0 && d.Hin > 0 && d.Win > 0 && d.Hout > 0 && d.Wout > 0 && d.N > 0,
                "ccvpe_igemm: bad shape B=%d in=%dx%d out=%dx%d N=%d", d.B, d.Hin, d.Win, d.Hout, d.Wout, d.N);
  CCVPE_REQUIRE(d.c0 > 0 && d.c0 % 8 == 0 && d.c1 >= 0 && d.c1 % 8 == 0 && d.ld0 >= d.c0 && d.ld0 % 8 == 0,
                "ccvpe_igemm: channel counts must be positive multiples of 8 (c0=%d ld0=%d c1=%d)", d.c0, d.ld0, d.c1);
  CCVPE_REQUIRE(d.c1 == 0 || (d.a1 && d.ld1 >= d.c1 && d.ld1 % 8 == 0), "ccvpe_igemm: bad second source");
  CCVPE_REQUIRE(d.stride >= 1 && d.kh >= 1 && d.kw >= 1 && d.kh * d.kw <= 9 && d.pad >= 0, "ccvpe_igemm: bad window");
  CCVPE_REQUIRE(!d.row_r1 || d.r1_w, "ccvpe_igemm: row_r1 needs r1_w");
  CCVPE_REQUIRE(d.relu == 0 || d.relu == 1, "ccvpe_igemm: relu must be 0 or 1");
  CCVPE_REQUIRE(d.out_mode >= 0 && d.out_mode <= 2, "ccvpe_igemm: bad out_mode %d", d.out_mode);
  CCVPE_REQUIRE(d.out_mode != 2 || d.out_dtype == CCVPE_F32, "ccvpe_igemm: planar output must be fp32");
  CCVPE_REQUIRE(d.out_mode != 1 || (d.N % 4 == 0 && (d.N / 4) % 8 == 0), "ccvpe_igemm: pixel-shuffle needs N = 4*Cout, Cout%%8==0");
  CCVPE_REQUIRE(d.out_mode == 2 || d.ldo >= (d.out_mode == 1 ? d.N / 4 : d.N), "ccvpe_igemm: ldo too small");
  CCVPE_REQUIRE(aligned16(d.a0) && aligned16(d.a1) && aligned16(d.out), "ccvpe_igemm: pointers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int backend = d.backend;
  if (backend == CCVPE_BACKEND_AUTO)
    backend = (d.dtype == CCVPE_BF16 && d.w_nk && igemm_tcgen05_supported(d)) ? CCVPE_BACKEND_TCGEN05
                                                                               : CCVPE_BACKEND_SIMT;
  if (backend == CCVPE_BACKEND_TCGEN05) {
    // wide shallow 3x3 levels take the row-ring kernel
    if (conv_ring_supported(d)) return conv_ring_tcgen05(d, st);
    return igemm_tcgen05(d, st, nullptr);
  }
  if (backend == CCVPE_BACKEND_SIMT) return igemm_simt(d, st);
  return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_igemm: unknown backend %d", d.backend);
}
