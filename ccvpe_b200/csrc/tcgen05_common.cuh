// Shared pieces of the tcgen05 kernels: PTX wrappers (mbarrier, TMA, tcgen05.mma / ld / commit), the shared-memory
// matrix descriptor, the common epilogue (TMEM -> registers -> bias / row-scale / rank-1 / ReLU -> global stores)
// and the host-side tensor-map encoder.  sm_100a only.
#pragma once

#include <cuda.h>

#include <cstdlib>
#include <mutex>

#include "common.cuh"

namespace ccvpe {

constexpr int TC_BM = 128;          // pixels per tile (UMMA M)
constexpr int TC_MAX_N = 256;       // widest accumulator tile (TMEM columns per stage)
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_EPI_THREADS = 32 * TC_EPI_WARPS;

// ---- PTX wrappers ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// True in exactly one lane of a converged warp.  Issuing the warp-level tcgen05 / TMA instructions under this predicate
// (instead of `lane == 0` inside a divergent branch) lets ptxas emit them straight on the uniform datapath; with a
// divergent single lane it wraps every UTCHMMA / UTMALDG / UTCBAR in an ELECT + BRA.U.ANY retry loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();  // ~2 s: a pipeline protocol bug must not hang the device
  }
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled shared-memory matrix descriptor.  A K block of kw bf16 channels is one swizzle row of 2*kw bytes
// (kw = 64 -> SWIZZLE_128B, 32 -> SWIZZLE_64B, 16 -> SWIZZLE_32B); 8 rows form a group, groups are 16*kw bytes apart.
__host__ __device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, int kw) {
  const uint64_t layout = kw == 64 ? 2 : (kw == 32 ? 4 : 6);
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, 16-byte units
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major), 16 B
  d |= (uint64_t)((16 * kw) >> 4) << 32;     // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
  d |= layout << 61;
  return d;
}


// ---- epilogue ------------------------------------------------------------------------------------------------------
struct EpiParams {
  int N, HWo, Wout, Hout;
  const float* bias;
  const float* row_scale;
  const float* row_r1;
  const float* r1_w;
  int relu, out_mode, out_f32, ldo;
  void* out;
};

// Stages the per-column epilogue constants of the N tile [n0, n0 + block_n) into shared memory (all epilogue threads
// call): bias, rank-1 weights and -- so that the per-row store loop carries no index arithmetic -- the element offset of
// every 8-column group relative to the row's first output pixel (channel, plus the quadrant displacement of the k2 s2
// transposed conv's pixel shuffle).  SiLU (relu == 2) is evaluated as h + h*tanh(h) with h = x/2, so its bias is staged
// pre-halved.
__device__ __forceinline__ void epi_stage_vectors(const EpiParams& e, float* s_bias, float* s_r1w, int* s_off, int n0,
                                                  int block_n, int et, int epi_threads = TC_EPI_THREADS) {
  const float bscale = e.relu == 2 ? 0.5f : 1.f;
  for (int c = et; c < block_n; c += epi_threads) {
    const int n = n0 + c;
    s_bias[c] = (e.bias && n < e.N) ? bscale * __ldg(e.bias + n) : 0.f;
    s_r1w[c] = (e.row_r1 && n < e.N) ? __ldg(e.r1_w + n) : 0.f;
    if ((c & 7) == 0) {
      int off = n;
      if (e.out_mode == 1) {
        const int cout = e.N >> 2;
        const int ij = n / cout, co = n - ij * cout;
        off = (ij >> 1) * 2 * e.Wout * e.ldo + (ij & 1) * e.ldo + co;
      }
      s_off[c >> 3] = off;
    }
  }
  asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
}

// Element offset of the first output pixel of accumulator row m (m = flattened (b, h, w) of the GEMM's M axis).
template <int MODE>
__device__ __forceinline__ int64_t epi_row_base(const EpiParams& e, int m) {
  if (MODE == 1) {   // pixel shuffle: pixel (q = b*H + h, w) -> (2q, 2w) of the [B*2H, 2W] output
    const int q = m / e.Wout, w = m - q * e.Wout;
    return ((int64_t)q * 4 * e.Wout + 2 * w) * e.ldo;
  }
  return (int64_t)m * e.ldo;
}

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// One thread = one accumulator row.  `halves` = number of warps sharing a TMEM lane group (each takes every
// `halves`-th 32-column chunk, starting at `half`).  taddr = TMEM address of (lane group, first column of the stage).
// Specialised at compile time on (output mode, rank-1 term, fp32 output); the kernels are instantiated once per variant.
//   MODE 0 channels-last | 1 pixel shuffle | 2 planar fp32 NCHW | 3 channels-last bf16 with SiLU
// bf16 outputs take the lean path: per 8 columns two LDS.128 (bias), 8 FFMA (+8 FMNMX or the SiLU), 4 F2FP, one LDS (group
// offset) and ONE 16-byte store -- the host guarantees 8-column groups never straddle N / a quadrant and 16-byte alignment
// (tc_epilogue_supported).  The epilogue, not the tensor pipe, bounds the shallow-K layers, so its instruction count is
// what is being minimised here.  row_base = epi_row_base() of the row (m_glob itself is only used by the planar mode).
// release_bar (an mbarrier address, or 0): arrived on by lane 0 as soon as the last TMEM chunk of the row is in registers,
// so the MMA issuer gets the accumulator stage back before the stores have drained.
template <int MODE, bool HAS_R1, bool OUT_F32>
__device__ __forceinline__ void epi_store_row(const EpiParams& e, uint32_t taddr, int half, int block_n, int n0,
                                              bool valid, int m_glob, int64_t row_base, float rs, float r1,
                                              const float* s_bias, const float* s_r1w, const int* s_off, int halves,
                                              uint32_t release_bar = 0) {
  const int lane = threadIdx.x & 31;
  const int N = e.N;
  const int ncols = min(block_n, N - n0);               // accumulator columns of this tile that exist
  const float lower = e.relu ? 0.f : -INFINITY;          // branch-free ReLU
  if (MODE == 3) rs *= 0.5f;

  auto process = [&](const uint32_t (&v)[32], int c0) {
    if (!valid) return;
#pragma unroll
    for (int g8 = 0; g8 < 4; ++g8) {
      const int cl = c0 + g8 * 8;             // column within the tile
      if (cl >= ncols) break;
      const float4 b0 = *reinterpret_cast<const float4*>(&s_bias[cl]);
      const float4 b1 = *reinterpret_cast<const float4*>(&s_bias[cl + 4]);
      float y[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      if (HAS_R1) {
        const float4 w0 = *reinterpret_cast<const float4*>(&s_r1w[cl]);
        const float4 w1 = *reinterpret_cast<const float4*>(&s_r1w[cl + 4]);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = fmaf(r1, wv[j], y[j]);
      }
      if (MODE == 3) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float h = fmaf(__uint_as_float(v[g8 * 8 + j]), rs, y[j]);
          y[j] = fmaf(h, tanh_approx(h), h);               // SiLU(x) = x * sigmoid(x) = h + h * tanh(h), h = x / 2
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = fmaxf(fmaf(__uint_as_float(v[g8 * 8 + j]), rs, y[j]), lower);
      }
      if (MODE == 2) {
        const int n = n0 + cl;
        float* o = static_cast<float*>(e.out) + (int64_t)(m_glob / e.HWo) * N * e.HWo + (m_glob % e.HWo);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (n + j < N) o[(int64_t)(n + j) * e.HWo] = y[j];
      } else if (OUT_F32) {
        const int n = n0 + cl;
        float* o = static_cast<float*>(e.out) + row_base + n;
        if ((n + 8 <= N) && ((e.ldo & 3) == 0)) {
          *reinterpret_cast<float4*>(o) = make_float4(y[0], y[1], y[2], y[3]);
          *reinterpret_cast<float4*>(o + 4) = make_float4(y[4], y[5], y[6], y[7]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (n + j < N) o[j] = y[j];
        }
      } else {
        __nv_bfloat16* o = static_cast<__nv_bfloat16*>(e.out) + (row_base + s_off[cl >> 3]);
        __nv_bfloat162 q0 = __floats2bfloat162_rn(y[0], y[1]), q1 = __floats2bfloat162_rn(y[2], y[3]);
        __nv_bfloat162 q2 = __floats2bfloat162_rn(y[4], y[5]), q3 = __floats2bfloat162_rn(y[6], y[7]);
        uint4 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&q0);
        pk.y = *reinterpret_cast<uint32_t*>(&q1);
        pk.z = *reinterpret_cast<uint32_t*>(&q2);
        pk.w = *reinterpret_cast<uint32_t*>(&q3);
        *reinterpret_cast<uint4*>(o) = pk;
      }
    }
  };

  // the accumulator stage goes back to the MMA issuer as soon as its last chunk is in registers
  auto release = [&]() {
    if (release_bar) {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(release_bar);
    }
  };

  // TMEM -> registers, double buffered: the load of the next chunk is in flight while this one is processed
  uint32_t va[32], vb2[32];
  const int cfirst = half * 32, cstep = 32 * halves;
  if (cfirst < block_n) tmem_ld32(taddr + (uint32_t)cfirst, va);
  else release();
  for (int c0 = cfirst; c0 < block_n; c0 += 2 * cstep) {
    tmem_ld_wait();
    const bool more1 = (c0 + cstep < block_n);
    if (more1) tmem_ld32(taddr + (uint32_t)(c0 + cstep), vb2);
    else release();
    process(va, c0);
    if (more1) {
      tmem_ld_wait();
      if (c0 + 2 * cstep < block_n) tmem_ld32(taddr + (uint32_t)(c0 + 2 * cstep), va);
      else release();
      process(vb2, c0 + cstep);
    }
  }
}

// Staged variant for the HBM-bound (shallow-K) layers, bf16 outputs only.  32 threads each storing their own row touch 32
// different 128-byte lines per instruction, which caps a row-per-thread epilogue at ~2.4 TB/s on B200
// (scripts/store_probe.cu).  Here every 32-column chunk (64 bytes per row) goes through a per-warp shared-memory tile
// instead (row pitch 80 bytes = an odd number of 16-byte units: the row-per-thread writes are bank-conflict free) and is
// copied out with 4 lanes per row / 8 rows per instruction, so consecutive pixels leave as contiguous runs (6 TB/s in the
// same probe).  Rows outside the problem are computed like the others and dropped at the copy (no divergent math).
// `stage` / `s_rowbase`: THIS WARP's 32 x 80-byte tile and 32 row offsets (16-byte units).  Single-buffered TMEM loads keep the register
// count low enough for 16 epilogue warps per SM, which is what hides the instruction latencies of this code.
constexpr int EPI_CHUNK_PITCH = 80;
constexpr int EPI_WARP_STAGE_BYTES = 32 * EPI_CHUNK_PITCH;

template <int MODE, bool HAS_R1>
__device__ __forceinline__ void epi_store_row_staged(const EpiParams& e, uint32_t taddr, int half, int halves, int block_n,
                                                     int n0, bool valid, int64_t row_base, float rs, float r1,
                                                     const float* s_bias, const float* s_r1w, const int* s_off,
                                                     uint32_t release_bar, uint8_t* stage, int32_t* s_rowbase) {
  const int lane = threadIdx.x & 31;
  const int ncols = min(block_n, e.N - n0);
  const float lower = e.relu ? 0.f : -INFINITY;
  if (MODE == 3) rs *= 0.5f;
  // row offsets travel as 32-bit indices of 16-byte units (outputs < 32 GB, checked on the host): one IMAD.WIDE per store
  s_rowbase[lane] = valid ? (int32_t)(row_base >> 3) : -1;
  uint8_t* my = stage + lane * EPI_CHUNK_PITCH;
  uint4* out16 = static_cast<uint4*>(e.out);
  const int cstep = 32 * halves;
  const int fr = lane >> 2, fc = lane & 3;          // copy-out role: row within a group of 8, 16-byte unit within the chunk
  const uint8_t* src = stage + fr * EPI_CHUNK_PITCH + fc * 16;
  auto release = [&]() {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(release_bar);
  };
  int c0 = half * 32;
  if (c0 >= ncols) release();
  for (; c0 < ncols; c0 += cstep) {
    uint32_t v[32];
    tmem_ld32(taddr + (uint32_t)c0, v);
    tmem_ld_wait();
    if (c0 + cstep >= ncols) release();             // that was this warp's last chunk of the accumulator stage
    auto group = [&](int g8) {                       // 8 columns: bias / rank-1 / scale / activation -> 16 staged bytes
      const int cl = c0 + g8 * 8;
      const float4 b0 = *reinterpret_cast<const float4*>(&s_bias[cl]);
      const float4 b1 = *reinterpret_cast<const float4*>(&s_bias[cl + 4]);
      float y[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      if (HAS_R1) {
        const float4 w0 = *reinterpret_cast<const float4*>(&s_r1w[cl]);
        const float4 w1 = *reinterpret_cast<const float4*>(&s_r1w[cl + 4]);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = fmaf(r1, wv[j], y[j]);
      }
      if (MODE == 3) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float h = fmaf(__uint_as_float(v[g8 * 8 + j]), rs, y[j]);
          y[j] = fmaf(h, tanh_approx(h), h);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = fmaxf(fmaf(__uint_as_float(v[g8 * 8 + j]), rs, y[j]), lower);
      }
      __nv_bfloat162 q0 = __floats2bfloat162_rn(y[0], y[1]), q1 = __floats2bfloat162_rn(y[2], y[3]);
      __nv_bfloat162 q2 = __floats2bfloat162_rn(y[4], y[5]), q3 = __floats2bfloat162_rn(y[6], y[7]);
      uint4 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&q0);
      pk.y = *reinterpret_cast<uint32_t*>(&q1);
      pk.z = *reinterpret_cast<uint32_t*>(&q2);
      pk.w = *reinterpret_cast<uint32_t*>(&q3);
      *reinterpret_cast<uint4*>(my + g8 * 16) = pk;
    };
    if (c0 + 32 <= ncols) {                           // full chunk: straight-line code
      group(0);
      group(1);
      group(2);
      group(3);
    } else {
#pragma unroll
      for (int g8 = 0; g8 < 4; ++g8)
        if (c0 + g8 * 8 < ncols) group(g8);
    }
    __syncwarp();
    const bool unit_ok = fc < ((min(32, ncols - c0)) >> 3);
    const int goff = unit_ok ? (s_off[(c0 >> 3) + fc] >> 3) : 0;
#pragma unroll
    for (int pass = 0; pass < 4; ++pass) {
      const int32_t rb = s_rowbase[pass * 8 + fr];
      const uint4 val = *reinterpret_cast<const uint4*>(src + pass * 8 * EPI_CHUNK_PITCH);
      if (unit_ok && rb >= 0) out16[(uint32_t)(rb + goff)] = val;
    }
    __syncwarp();
  }
}

// bf16 outputs use 16-byte stores of 8-column groups: channel counts / strides must be multiples of 8, base 16-B aligned.
inline bool tc_epilogue_supported(const ccvpe_igemm_desc& d) {
  if (d.out_dtype != CCVPE_BF16) return true;
  if (d.out_mode == 2) return false;
  const int cout = d.out_mode == 1 ? d.N / 4 : d.N;
  // (the staged epilogue addresses the output with 32-bit indices of 16-byte units: keep it below 16 GB, padding included)
  const int64_t out_elems = (int64_t)(d.out_mode == 1 ? 4 : 1) * d.B * d.Hout * d.Wout * d.ldo;
  return (cout % 8 == 0) && (d.ldo % 8 == 0) && ((reinterpret_cast<uintptr_t>(d.out) & 15) == 0) &&
         (d.out_mode != 1 || d.N % 4 == 0) && out_elems < (1LL << 33);
}

// Epilogue variant of a descriptor: 0 conv bf16 | 1 conv bf16 + rank-1 | 2 conv fp32 channels-last | 3 planar fp32 |
// 4 pixel-shuffle bf16 | 5 pixel-shuffle bf16 + rank-1 | 6 channels-last bf16 + SiLU (generic igemm kernel only).
// CCVPE_EPI_SWITCH expands `X(MODE, HAS_R1, OUT_F32)` for variants 0..5.
inline int epi_variant(const EpiParams& e) {
  if (e.relu == 2) return 6;
  if (e.out_mode == 1) return e.row_r1 ? 5 : 4;
  if (e.out_mode == 2) return 3;
  if (e.out_f32) return 2;
  return e.row_r1 ? 1 : 0;
}
#define CCVPE_EPI_SWITCH(variant, X) \
  switch (variant) {                 \
    case 0: X(0, false, false); break; \
    case 1: X(0, true, false); break;  \
    case 2: X(0, false, true); break;  \
    case 3: X(2, false, true); break;  \
    case 4: X(1, false, false); break; \
    default: X(1, true, false); break; \
  }

// ---- host side ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &sym, 12000, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

inline int encode_map(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box, int kw) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(CCVPE_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  kw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (kw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(CCVPE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rank=%d dims=[%llu,%llu,%llu,..] box=[%u,%u,%u,..]",
                (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
                (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], box[1], rank > 2 ? box[2] : 0);
  return CCVPE_OK;
}


// K-block width (bf16 channels) used for a source with c channels; one block is one swizzle row of 2*width bytes.
// Narrow sources get narrow blocks so TMA neither over-fetches nor zero-fills most of the tile (include/ccvpe_b200.h
// documents the same rule for the w_nk weight layout; ccvpe_b200/cabi.py:w_nk_layout builds it).
// 33..63 channels take ONE 64-wide block rather than two 32-wide ones: the padded K extent (64), the shared-memory
// footprint and the number of K16 MMA slices are the same, but TMA walks half as many box rows (its cost is per box row).
inline int tc_block_width(int c) { return c <= 16 ? 16 : (c <= 32 ? 32 : 64); }

inline void fill_epi(EpiParams& e, const ccvpe_igemm_desc& d) {
  e.N = d.N;
  e.HWo = d.Hout * d.Wout;
  e.Wout = d.Wout;
  e.Hout = d.Hout;
  e.bias = d.bias;
  e.row_scale = d.row_scale;
  e.row_r1 = d.row_r1;
  e.r1_w = d.r1_w;
  e.relu = d.relu;
  e.out_mode = d.out_mode;
  e.out_f32 = (d.out_dtype == CCVPE_F32);
  e.ldo = d.ldo;
  e.out = d.out;
}

}  // namespace ccvpe
