// Weight gradient of the 3x3 convolutions on tensor cores (training step, BASELINE.json configs[4]):
//
//   dW[tap][c][n] = sum_pix A[pix + shift(tap), c] * G[pix, n]            A = layer input, G = dY, both channels-last bf16
//
// As a GEMM the reduction axis is the PIXEL axis, which is the slow axis of both channels-last operands -- so both UMMA
// operands are MN-major: a TMA box [channels x pixels] of a channels-last map lands in shared memory as one swizzle row per
// pixel, which is exactly the canonical MN-major layout (channels contiguous inside a row, consecutive K = consecutive
// rows, 8-row groups SBO apart, 64-/32-channel atoms LBO apart).  The very boxes the forward implicit GEMM loads as K-major
// tiles (K = channels) are re-interpreted here with K = pixels; only the matrix descriptors and two idesc bits differ.
//
// Tile: 128 output channels n (UMMA M) x 32 input channels c (UMMA N) x all 9 taps: nine accumulators [128 x 32] in TMEM
// (288 of 512 columns).  Per 64-pixel step the G tile [64 px x 128 n] is loaded ONCE, and so is the A tile: ONE halo box
// [(hb + 2) x (wb + 2) px x 32 c] (conv padding = TMA zero fill) serves all nine taps -- tap (ky, kx) of the 16 pixels of a
// K step is the same shared-memory tile read (ky * (wb + 2) + kx) rows further down, i.e. only the start address of the
// matrix descriptor moves (the swizzle is a function of the absolute shared-memory address, the one TMA wrote with).
// 36 MMAs of 128x32x16 per stage against ~260 TMA box rows (nine separate tap boxes would be 640: TMA issues ~3 cycles
// per box row, which is what bounded the first version of this kernel).  K (pixels) is split over
// CTAs when there are fewer tiles than SMs; partial tiles go to the workspace and are folded in a fixed order
// (deterministic).  Warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2-5 = epilogue.
#include "tcgen05_common.cuh"

namespace ccvpe {

constexpr int WT_BK = 64;          // pixels per pipeline stage
constexpr int WT_CT = 32;          // A-channel tile
constexpr int WT_NT = 128;         // G-channel tile
constexpr int WT_TAPS = 9;
constexpr int WT_THREADS = 192;
constexpr int WT_MAX_STAGES = 6;
constexpr int WT_G_BYTES = WT_BK * WT_NT * 2;          // 16 KB: two [64 px x 64 n] SWIZZLE_128B boxes
constexpr int WT_A_BYTES = WT_BK * WT_CT * 2;          // 4 KB per k2 s2 tap, SWIZZLE_64B
constexpr int WT_ROW_BYTES = WT_CT * 2;                // 64 B: one pixel of an A tile

struct WgradTcParams {
  CUtensorMap tm_a0, tm_a1, tm_g;
  int c0, c1, ctot, N, Q;
  int W, H, B, wb, hb, tiles_w, tiles_h;
  int ksteps_total, ksteps_per_split;
  int c_tiles0;
  int stages;
  int stage_bytes, a_tx;               // 3x3: one (hb+2) x (wb+2) A box per stage; a_tx = bytes TMA delivers for it
  int k2s2, taps;                      // k2 s2 layers: 4 taps gathered through a 5-D map [c][dw][j][dh][(b, i)]
  float* dst;
};

// MN-major shared-memory matrix descriptor: `lbo` = byte distance between swizzle atoms along M/N, `sbo` = byte distance
// between 8-row groups along K; layout 2 = SWIZZLE_128B, 4 = SWIZZLE_64B.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint64_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= layout << 61;
  return d;
}

__global__ void __launch_bounds__(WT_THREADS, 1) wgrad_tcgen05_kernel(const __grid_constant__ WgradTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[WT_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_empty[WT_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_acc;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;

  const int ct = blockIdx.x;
  const bool src1 = ct >= p.c_tiles0;
  const int c_start = (src1 ? ct - p.c_tiles0 : ct) * WT_CT;
  const int c_glob0 = (src1 ? p.c0 : 0) + c_start;
  const int c_valid = min(WT_CT, (src1 ? p.c1 : p.c0) - c_start);
  const int n0 = blockIdx.y * WT_NT;
  const int ks_begin = blockIdx.z * p.ksteps_per_split;
  const int ks_end = min(p.ksteps_total, ks_begin + p.ksteps_per_split);

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(&bar_acc), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(src1 ? &p.tm_a1 : &p.tm_a0);
    prefetch_tmap(&p.tm_g);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    const CUtensorMap* tma = src1 ? &p.tm_a1 : &p.tm_a0;
    // the second 64-channel G box of a tile whose N range ends inside the first re-reads the first (never fully out of
    // bounds); its accumulator rows are dropped by the epilogue
    const int n1 = (n0 + 64 < p.N) ? n0 + 64 : n0;
    int stage = 0;
    uint32_t phase = 0;
    const int per_img = p.tiles_w * p.tiles_h;
    for (int ks = ks_begin; ks < ks_end; ++ks) {
      // 3x3: (image, row block, column block) of the layer;  k2 s2: ((image, output row) block, output column block) --
      // p.H is then the number of merged (image, row) lines and one "image" covers them all
      const int b = ks / per_img, r = ks - b * per_img;
      const int th = r / p.tiles_w, tw = r - th * p.tiles_w;
      const int h0 = th * p.hb, w0 = tw * p.wb;
      const int m0 = (b * p.H + h0) * p.W + w0;            // first pixel of the block in the flattened G rows
      mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
      if (elect_one()) {
        const uint32_t full = smem_u32(&bar_full[stage]);
        const uint32_t dst = smem_base + (uint32_t)(stage * p.stage_bytes);
        mbar_arrive_expect_tx(full, (uint32_t)(WT_G_BYTES + (p.k2s2 ? p.taps * WT_A_BYTES : p.a_tx)));
        tma_load_2d(dst, &p.tm_g, full, n0, m0);
        tma_load_2d(dst + WT_G_BYTES / 2, &p.tm_g, full, n1, m0);
        if (p.k2s2) {
#pragma unroll
          for (int tap = 0; tap < 4; ++tap)      // tap = dh * 2 + dw
            tma_load_5d(dst + WT_G_BYTES + tap * WT_A_BYTES, tma, full, c_start, tap & 1, w0, tap >> 1, h0);
        } else {
          tma_load_4d(dst + WT_G_BYTES, tma, full, c_start, w0 - 1, h0 - 1, b);
        }
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // D[128 n x 96 (kx, c)] (+)= G^T[128 n x 16 px] * [A_(ky,0) | A_(ky,1) | A_(ky,2)][16 px x 96]; both operands MN-major
    // (idesc bits 15, 16).  The three kx taps of a ky row are three 32-channel atoms of ONE B operand: the same rows of
    // the halo tile shifted by one pixel (LBO = 64 B: overlapping atoms).
    // One thread issues everything, at ~5 cycles per dependent instruction, so the per-MMA descriptor words are
    // precomputed: 12 MMAs per stage, two adds each.
    constexpr int NW = 3 * WT_CT;                          // 96 accumulator columns per MMA
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(NW >> 3) << 17) |
                           ((uint32_t)(WT_NT >> 4) << 24);
    const int pitch = p.wb + 2;                            // pixels per row of the halo tile
    uint32_t a_off[WT_BK / 16][3];                         // 16-byte units from the stage base
#pragma unroll
    for (int kk = 0; kk < WT_BK / 16; ++kk) {
      const int hrow = (kk * 16) / p.wb, wcol = (kk * 16) - hrow * p.wb;   // the 16 pixels of K step kk: row hrow, from wcol
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
        a_off[kk][ky] = (uint32_t)(WT_G_BYTES + ((hrow + ky) * pitch + wcol) * WT_ROW_BYTES) >> 4;
    }
    const uint64_t gdesc0 = make_smem_desc_mn(smem_base, WT_G_BYTES / 2, 1024, 2);
    const uint64_t adesc0 = make_smem_desc_mn(smem_base, p.k2s2 ? WT_A_BYTES : WT_ROW_BYTES, 512, 4);
    // k2 s2: the two dw taps of a dh row are two atoms (4 KB apart) of one N = 64 MMA
    const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(2 * WT_CT >> 3) << 17) |
                            ((uint32_t)(WT_NT >> 4) << 24);
    const uint32_t stage_units = (uint32_t)p.stage_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t accumulate = 0;
    for (int ks = ks_begin; ks < ks_end; ++ks) {
      mbar_wait(smem_u32(&bar_full[stage]), phase);
      tc_fence_after();
      const uint32_t soff = (uint32_t)stage * stage_units;
      if (elect_one()) {
        if (p.k2s2) {
#pragma unroll
          for (int kk = 0; kk < WT_BK / 16; ++kk) {
            const uint64_t gdesc = gdesc0 + soff + (uint32_t)(kk * (2048 >> 4));
#pragma unroll
            for (int dh = 0; dh < 2; ++dh)
              umma_bf16(tmem_base + (uint32_t)(dh * 2 * WT_CT), gdesc,
                        adesc0 + soff + (uint32_t)((WT_G_BYTES + dh * 2 * WT_A_BYTES + kk * 1024) >> 4), idesc2,
                        (kk == 0) ? accumulate : 1u);
          }
        } else {
#pragma unroll
          for (int kk = 0; kk < WT_BK / 16; ++kk) {
            const uint64_t gdesc = gdesc0 + soff + (uint32_t)(kk * (2048 >> 4));   // 16 pixels of 128-byte rows per K step
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
              umma_bf16(tmem_base + (uint32_t)(ky * NW), gdesc, adesc0 + soff + a_off[kk][ky], idesc,
                        (kk == 0) ? accumulate : 1u);
          }
        }
        umma_commit(smem_u32(&bar_empty[stage]));
      }
      accumulate = 1;
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
    if (elect_one()) umma_commit(smem_u32(&bar_acc));
    __syncwarp();
  } else {
    // ===================== epilogue: TMEM -> out[tap][c][n] (n contiguous: one 128-byte line per warp and channel) ====
    const int lg = warp & 3;                                   // TMEM lane group this warp may read
    const int n = n0 + lg * 32 + lane;
    mbar_wait(smem_u32(&bar_acc), 0);
    tc_fence_after();
    const bool n_ok = n < p.N && (lg * 32 + lane < 64 || n0 + 64 < p.N);     // (rows 64.. duplicate rows 0.. on a short tile)
    for (int tap = 0; tap < p.taps; ++tap) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(tap * WT_CT), v);
      tmem_ld_wait();
      if (n_ok && ks_end > ks_begin) {
        float* o = p.dst + ((int64_t)blockIdx.z * p.Q + (int64_t)tap * p.ctot + c_glob0) * p.N + n;
#pragma unroll
        for (int c = 0; c < WT_CT; ++c)
          if (c < c_valid) o[(int64_t)c * p.N] = __uint_as_float(v[c]);
      } else if (n_ok) {
        float* o = p.dst + ((int64_t)blockIdx.z * p.Q + (int64_t)tap * p.ctot + c_glob0) * p.N + n;
        for (int c = 0; c < c_valid; ++c) o[(int64_t)c * p.N] = 0.f;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

int launch_reduce_splits(const float* ws, float* out, int64_t n, int splits, cudaStream_t st);   // train_ops.cu

// (3x3 stride-1 pad-1 convs, and k2 s2 convs -- the weight gradients of the transposed convs and of the aerial cell conv)
struct WgradTcPlan {
  bool k2s2;
  int wb, hb, tiles_w, tiles_h, ksteps, c_tiles0, c_tiles1, n_tiles, splits, ksteps_per_split;
};

static bool plan_wgrad_tc(const ccvpe_wgrad_desc& d, WgradTcPlan& pl) {
  if (d.dtype != CCVPE_BF16 || d.g_row_scale) return false;
  const bool conv3 = d.kh == 3 && d.kw == 3 && d.stride == 1 && d.pad == 1 && d.Hin == d.Hout && d.Win == d.Wout;
  const bool k2s2 = d.kh == 2 && d.kw == 2 && d.stride == 2 && d.pad == 0 && d.Hin == 2 * d.Hout && d.Win == 2 * d.Wout &&
                    d.c1 == 0;
  if (!conv3 && !k2s2) return false;
  if (d.c0 % 8 || d.c1 % 8 || d.ld0 % 8 || (d.c1 && d.ld1 % 8) || d.N % 8 || d.ldg % 8) return false;
  if (!aligned16(d.a0) || (d.c1 && !aligned16(d.a1)) || !aligned16(d.g)) return false;
  pl.k2s2 = k2s2;
  // pixel blocks of 64: 3x3 -> (wb x hb) pixels of one image; k2 s2 -> wb output columns x hb merged (image, row) lines
  const int W = d.Wout, H = k2s2 ? d.Hout * d.B : d.Hout;
  if (W >= WT_BK) {
    if (W % WT_BK) return false;
    pl.wb = WT_BK;
    pl.hb = 1;
  } else {
    if (WT_BK % W || H % (WT_BK / W)) return false;
    pl.wb = W;
    pl.hb = WT_BK / W;
  }
  pl.tiles_w = W / pl.wb;
  pl.tiles_h = H / pl.hb;
  pl.ksteps = (k2s2 ? 1 : d.B) * pl.tiles_w * pl.tiles_h;
  pl.c_tiles0 = (d.c0 + WT_CT - 1) / WT_CT;
  pl.c_tiles1 = (d.c1 + WT_CT - 1) / WT_CT;
  pl.n_tiles = (d.N + WT_NT - 1) / WT_NT;
  const int tiles = (pl.c_tiles0 + pl.c_tiles1) * pl.n_tiles;
  int splits = (sm_count() + tiles - 1) / tiles;
  const int max_splits = (pl.ksteps + 7) / 8;                // at least 8 pipeline steps per CTA
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  pl.ksteps_per_split = (pl.ksteps + splits - 1) / splits;
  pl.splits = (pl.ksteps + pl.ksteps_per_split - 1) / pl.ksteps_per_split;
  return true;
}

int wgrad_tcgen05_supported(const ccvpe_wgrad_desc& d) {
  WgradTcPlan pl;
  return plan_wgrad_tc(d, pl) ? 1 : 0;
}

int64_t wgrad_tcgen05_workspace_elems(const ccvpe_wgrad_desc& d) {
  WgradTcPlan pl;
  if (!plan_wgrad_tc(d, pl)) return 0;
  return pl.splits > 1 ? (int64_t)pl.splits * d.kh * d.kw * (d.c0 + d.c1) * d.N : 0;
}

int wgrad_tcgen05(const ccvpe_wgrad_desc& d, cudaStream_t st) {
  WgradTcPlan pl;
  if (!plan_wgrad_tc(d, pl)) return fail(CCVPE_ERR_UNSUPPORTED, "wgrad_tcgen05: unsupported shape");
  static thread_local WgradTcParams p;
  memset(&p, 0, sizeof(p));
  p.k2s2 = pl.k2s2 ? 1 : 0;
  p.taps = pl.k2s2 ? 4 : WT_TAPS;
  p.c0 = d.c0; p.c1 = d.c1; p.ctot = d.c0 + d.c1; p.N = d.N; p.Q = p.taps * p.ctot;
  p.W = d.Wout; p.H = pl.k2s2 ? d.Hout * d.B : d.Hout; p.B = pl.k2s2 ? 1 : d.B;
  p.wb = pl.wb; p.hb = pl.hb; p.tiles_w = pl.tiles_w; p.tiles_h = pl.tiles_h;
  p.ksteps_total = pl.ksteps; p.ksteps_per_split = pl.ksteps_per_split;
  p.c_tiles0 = pl.c_tiles0;
  p.a_tx = (pl.wb + 2) * (pl.hb + 2) * WT_ROW_BYTES;
  p.stage_bytes = pl.k2s2 ? WT_G_BYTES + p.taps * WT_A_BYTES : WT_G_BYTES + (p.a_tx + 1023) / 1024 * 1024;
  p.stages = WT_MAX_STAGES;
  while (p.stages * p.stage_bytes > 200 * 1024) --p.stages;
  const int64_t n_out = (int64_t)p.Q * d.N;
  if (pl.splits > 1) {
    if (!d.workspace || d.workspace_elems < (int64_t)pl.splits * n_out)
      return fail(CCVPE_ERR_BAD_ARGUMENT, "wgrad_tcgen05: workspace too small");
    p.dst = d.workspace;
  } else {
    p.dst = d.out;
  }
  int rc;
  if (pl.k2s2) {
    // [c][dw = 2][j = Wout][dh = 2][(b, i) = B * Hout]: output pixel ((b, i), j), tap (dh, dw) reads input pixel (2i + dh, 2j + dw)
    uint64_t dims[5] = {(uint64_t)d.c0, 2, (uint64_t)d.Wout, 2, (uint64_t)d.Hout * d.B};
    uint64_t str[4] = {(uint64_t)d.ld0 * 2, 2ull * d.ld0 * 2, (uint64_t)d.Win * d.ld0 * 2, 2ull * d.Win * d.ld0 * 2};
    uint32_t box[5] = {WT_CT, 1, (uint32_t)pl.wb, 1, (uint32_t)pl.hb};
    if ((rc = encode_map(&p.tm_a0, d.a0, 5, dims, str, box, 32)) != CCVPE_OK) return rc;
  }
  for (int s = 0; s < ((d.c1 ? 2 : 1) * (pl.k2s2 ? 0 : 1)); ++s) {
    const void* base = s ? d.a1 : d.a0;
    const int c = s ? d.c1 : d.c0, ld = s ? d.ld1 : d.ld0;
    uint64_t dims[4] = {(uint64_t)c, (uint64_t)d.Win, (uint64_t)d.Hin, (uint64_t)d.B};
    uint64_t str[3] = {(uint64_t)ld * 2, (uint64_t)d.Win * ld * 2, (uint64_t)d.Hin * d.Win * ld * 2};
    uint32_t box[4] = {WT_CT, (uint32_t)(pl.wb + 2), (uint32_t)(pl.hb + 2), 1};
    if ((rc = encode_map(s ? &p.tm_a1 : &p.tm_a0, base, 4, dims, str, box, 32)) != CCVPE_OK) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)d.N, (uint64_t)d.B * d.Hout * d.Wout};
    uint64_t str[1] = {(uint64_t)d.ldg * 2};
    uint32_t box[2] = {64, WT_BK};
    if ((rc = encode_map(&p.tm_g, d.g, 2, dims, str, box, 64)) != CCVPE_OK) return rc;
  }
  const int smem = p.stages * p.stage_bytes + 1024;
  static thread_local uint64_t attr_set = 0;
  if (first_use_on_device(attr_set)) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 4096);
    if (e != cudaSuccess) return fail(CCVPE_ERR_CUDA, "cudaFuncSetAttribute(wgrad): %s", cudaGetErrorString(e));
  }
  const dim3 grid(pl.c_tiles0 + pl.c_tiles1, pl.n_tiles, pl.splits);
  wgrad_tcgen05_kernel<<<grid, WT_THREADS, smem, st>>>(p);
  rc = check_launch("wgrad_tcgen05_kernel");
  if (rc != CCVPE_OK) return rc;
  if (pl.splits > 1) rc = launch_reduce_splits(d.workspace, d.out, n_out, pl.splits, st);
  return rc;
}

}  // namespace ccvpe
