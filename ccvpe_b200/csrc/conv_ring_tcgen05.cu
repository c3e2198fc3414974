// Row-ring 3x3 convolution on tcgen05 -- the path for the wide, shallow decoder levels (W >= 128, C <= ~100), which
// are HBM-bound and where the generic per-tap pipeline is limited by TMA's per-row issue rate (measured on B200:
// ~3.5 cycles per box row, scripts/tma_probe.cu) and by one barrier round trip per tiny K block.
//
// A CTA walks a 128-pixel-wide strip of one image downwards.  Every INPUT row segment (130 pixels: the strip plus a
// one-pixel halo, out-of-image pixels are TMA zero fill) is loaded ONCE into a ring of shared-memory row slots; the nine
// taps of an output row are nine shifted views of three ring slots: tap (dy, dx) reads slot(y + dy - 1) starting dx
// rows into the tile, which for the dense K-major swizzled layout is just a start-address offset of the UMMA
// descriptor (the swizzle XOR is a function of the absolute shared-memory address, the same one TMA used to write).
// All weights of the layer stay resident in shared memory, so the steady state is: 1 TMA row load, 1 barrier wait,
// 9 x blocks MMAs, 1 commit per 128 output pixels, and HBM/L2 traffic of exactly one read of the input.
//
// Warp roles and the epilogue are the same as in igemm_tcgen05.cu (shared through tcgen05_common.cuh).
#include "tcgen05_common.cuh"

namespace ccvpe {

constexpr int RING_THREADS = 192;     // warp 0 producer, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue
constexpr int RING_EPI_THREADS = 128;
constexpr int RING_MAX_DEPTH = 8;
constexpr int RING_HALO_W = TC_BM + 2;
constexpr int RING_SMEM_BUDGET = 208 * 1024;
constexpr int RING_MAX_STEPS = 4;     // K16 slices per tap of the unrolled issue path (4 x 16 = 64 padded input channels)

struct RingParams {
  CUtensorMap tm_a0, tm_a1, tm_b0, tm_b1;
  int nb0, nb1, c0, c1, kw0, kw1, kpad0, kpad1;
  int block_n, depth, tmem_cols;
  int B, H, W, strips, R, chunks, total_units;
  int a_blk0, a_blk1, row_bytes;      // ring slot geometry
  int w_blk0, w_blk1, w_tap_bytes;    // resident weight geometry
  int tx_row, tx_weights;
  // Unrolled issue path (NS > 0): one entry per K16 slice of a tap, precomputed on the host so that the single MMA-issuing
  // thread forms every descriptor with one add from the constant bank: descriptor high word (swizzle mode + group stride),
  // A offset of (slice, dx) inside a ring row and B offset of (tap, slice) inside the resident weights, all in 16-byte
  // descriptor units.
  int n_steps, unrolled;
  uint32_t st_hi[RING_MAX_STEPS], st_adx[RING_MAX_STEPS][3], st_wt[9][RING_MAX_STEPS];
  EpiParams e;
};


// STAGE_OUT: bf16 rows leave through per-warp staging tiles (tiles of >= 32 columns; for 16-column tiles the direct
// 32-byte stores measure faster, and compiling both paths into one kernel spills).
// NS > 0: the layer's taps have exactly NS K16 slices and the MMA issue sequence of an output row is straight-line code
// (see the issuer below); NS == 0: generic loops.
// These variants also run TWO epilogue groups of four warps, one per TMEM accumulator stage (even / odd output rows): with
// the issue stream shortened, a single group's ~340 dependent instructions per row were the next limit.
template <int MODE, bool HAS_R1, bool OUT_F32, bool STAGE_OUT, int NS = 0>
__global__ void __launch_bounds__(NS > 0 ? RING_THREADS + RING_EPI_THREADS : RING_THREADS, NS > 0 ? 2 : 3) conv_ring_tcgen05_kernel(const __grid_constant__ RingParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[RING_MAX_DEPTH];
  __shared__ __align__(8) uint64_t bar_empty[RING_MAX_DEPTH];
  __shared__ __align__(8) uint64_t bar_w;
  __shared__ __align__(8) uint64_t bar_tmem_full[2];
  __shared__ __align__(8) uint64_t bar_tmem_empty[2];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float s_bias[TC_MAX_N];
  __shared__ __align__(16) float s_r1w[TC_MAX_N];
  __shared__ int s_off[TC_MAX_N / 8];
  // bf16 rows leave through per-warp staging tiles (coalesced copy-out, see epi_store_row_staged)
  constexpr bool STAGED = STAGE_OUT && !OUT_F32 && MODE != 2;
  constexpr int EPI_GROUPS = NS > 0 ? 2 : 1;
  __shared__ __align__(16) uint8_t s_stage[STAGED ? EPI_GROUPS * 4 * EPI_WARP_STAGE_BYTES : 16];
  __shared__ int32_t s_rowbase[STAGED ? EPI_GROUPS * TC_BM : 1];
  __shared__ __align__(16) uint4 s_blk[4];   // per K block: descriptor offsets (16-byte units) for the MMA issuer

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t w_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t ring_base = w_base + 9u * (uint32_t)p.w_tap_bytes;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.depth; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(&bar_w), 1);
    {
      uint32_t ao = 0, wo = 0;
      for (int g = 0; g < p.nb0 + p.nb1; ++g) {
        const bool s1 = g >= p.nb0;
        const int kw = s1 ? p.kw1 : p.kw0, cb = s1 ? g - p.nb0 : g, c = s1 ? p.c1 : p.c0, nb = s1 ? p.nb1 : p.nb0;
        const uint32_t nk16 = (cb == nb - 1) ? (uint32_t)((c - cb * kw + 15) >> 4) : (uint32_t)(kw >> 4);
        s_blk[g] = make_uint4(ao >> 4, wo >> 4, (uint32_t)(make_smem_desc(0, kw) >> 32),
                              ((uint32_t)(kw * 2) >> 4) | (nk16 << 16));
        ao += s1 ? p.a_blk1 : p.a_blk0;
        wo += s1 ? p.w_blk1 : p.w_blk0;
      }
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tmem_full[a]), 1);
      mbar_init(smem_u32(&bar_tmem_empty[a]), RING_EPI_THREADS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tm_a0);
    prefetch_tmap(&p.tm_b0);
    if (p.nb1) {
      prefetch_tmap(&p.tm_a1);
      prefetch_tmap(&p.tm_b1);
    }
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged, single-lane issue via elect_one) =====================
    {
      if (elect_one()) {   // all weights of the layer, once
        mbar_arrive_expect_tx(smem_u32(&bar_w), (uint32_t)p.tx_weights);
        for (int tap = 0; tap < 9; ++tap) {
          uint32_t dst = w_base + (uint32_t)(tap * p.w_tap_bytes);
          const int kcol = tap * (p.kpad0 + p.kpad1);
          for (int cb = 0; cb < p.nb0; ++cb, dst += p.w_blk0) tma_load_2d(dst, &p.tm_b0, smem_u32(&bar_w), kcol + cb * p.kw0, 0);
          for (int cb = 0; cb < p.nb1; ++cb, dst += p.w_blk1)
            tma_load_2d(dst, &p.tm_b1, smem_u32(&bar_w), kcol + p.kpad0 + cb * p.kw1, 0);
        }
      }
      __syncwarp();
      int slot = 0;
      uint32_t phase = 0;
      for (int unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
        const int rc = unit % p.chunks;
        const int xs = (unit / p.chunks) % p.strips;
        const int b = unit / (p.chunks * p.strips);
        const int y0 = rc * p.R, x0 = xs * TC_BM;
        const int y_lo = y0 > 0 ? y0 - 1 : 0;
        const int y_hi = (y0 + p.R < p.H) ? y0 + p.R : p.H - 1;
        for (int y = y_lo; y <= y_hi; ++y) {
          mbar_wait(smem_u32(&bar_empty[slot]), phase ^ 1u);
          if (elect_one()) {
            const uint32_t full = smem_u32(&bar_full[slot]);
            mbar_arrive_expect_tx(full, (uint32_t)p.tx_row);
            uint32_t dst = ring_base + (uint32_t)(slot * p.row_bytes);
            const int yrow = b * p.H + y;
            for (int cb = 0; cb < p.nb0; ++cb, dst += p.a_blk0) tma_load_3d(dst, &p.tm_a0, full, cb * p.kw0, x0 - 1, yrow);
            for (int cb = 0; cb < p.nb1; ++cb, dst += p.a_blk1) tma_load_3d(dst, &p.tm_a1, full, cb * p.kw1, x0 - 1, yrow);
          }
          __syncwarp();
          if (++slot == p.depth) {
            slot = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // One thread issues every MMA, so its instruction count per output row IS the kernel's clock for the narrow levels:
    // everything is precomputed into registers (16-byte-unit descriptor offsets per K block), ring slots roll without
    // div/mod, and the (block, dx, k) loops are fully unrolled.
    {  // the whole warp runs the loop converged; single-lane work is predicated with elect_one()
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.block_n >> 3) << 17) |
                             ((uint32_t)(TC_BM >> 4) << 24);
      const int nblk = p.nb0 + p.nb1;
      const uint32_t lo_flag = 1u << 16;
      const uint32_t ring16 = ((ring_base & 0x3FFFFu) >> 4) | lo_flag, row16 = (uint32_t)p.row_bytes >> 4;
      const uint32_t w16 = ((w_base & 0x3FFFFu) >> 4) | lo_flag, tap16 = (uint32_t)p.w_tap_bytes >> 4;
      const int depth = p.depth, H = p.H, R = p.R, chunks = p.chunks;
      const uint32_t bar_full0 = smem_u32(&bar_full[0]), bar_empty0 = smem_u32(&bar_empty[0]);
      const uint32_t bar_tf0 = smem_u32(&bar_tmem_full[0]), bar_te0 = smem_u32(&bar_tmem_empty[0]);
      // fast path for a single 16-channel K block (all four 512x512 convs): everything in registers
      const bool simple = (nblk == 1) && ((s_blk[0].w >> 16) == 1u);
      const uint64_t simple_hi = (uint64_t)s_blk[0].z << 32;
      const uint32_t simple_a = s_blk[0].x, simple_rowp = s_blk[0].w & 0xFFFFu;
      uint32_t simple_w[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) simple_w[t] = w16 + (uint32_t)t * tap16 + s_blk[0].y;
      mbar_wait(smem_u32(&bar_w), 0);
      tc_fence_after();
      // ring position of the NEXT row to be consumed for the first time (same sequence as the producer)
      int nslot = 0;
      uint32_t nphase = 0;
      int it = 0;
      for (int unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
        const int y0 = (unit % chunks) * R;
        // slots of input rows yo-1, yo, yo+1 (-1: outside the image, never loaded)
        int s_prev = -1, s_cur = -1, s_next = -1;
        auto acquire = [&]() {   // waits for the next ring row and returns its slot
          const int sl = nslot;
          mbar_wait(bar_full0 + 8u * (uint32_t)sl, nphase);
          if (++nslot == depth) {
            nslot = 0;
            nphase ^= 1u;
          }
          return sl;
        };
        if (y0 > 0) s_prev = acquire();
        s_cur = acquire();
        for (int yo = y0; yo < y0 + R; ++yo, ++it) {
          s_next = (yo + 1 < H) ? acquire() : -1;
          tc_fence_after();
          const uint32_t acc = (uint32_t)it & 1u;
          mbar_wait(bar_te0 + 8u * acc, (((uint32_t)it >> 1) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + acc * (uint32_t)p.block_n;
          if (NS > 0) {
            // Measured (ncu source view of the generic loop on the 40 -> 40 level-2 conv): the issuing warp executed 465
            // instructions per output row for 27 MMAs and was never waiting -- its own instruction stream was the
            // kernel's clock (3000 cycles per row).  Here the (dy, slice, dx) nest is fully unrolled and every
            // descriptor is one add of a constant-bank entry to a per-row base.
            if (elect_one()) {
              uint32_t accumulate = 0;
#pragma unroll
              for (int dy = 0; dy < 3; ++dy) {
                const int sl = dy == 0 ? s_prev : (dy == 1 ? s_cur : s_next);
                if (sl >= 0) {
                  const uint32_t a_row = ring16 + (uint32_t)sl * row16;
#pragma unroll
                  for (int j = 0; j < NS; ++j) {
                    const uint64_t hi = (uint64_t)p.st_hi[j] << 32;
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) {
                      umma_bf16(tmem_d, hi | (a_row + p.st_adx[j][dx]), hi | (w16 + p.st_wt[dy * 3 + dx][j]), idesc, accumulate);
                      accumulate = 1;
                    }
                  }
                }
              }
            }
            __syncwarp();
          } else if (simple) {
            // one 16-channel K block (the 512^2 level): nine MMAs, every descriptor word precomputed
            if (elect_one()) {
              uint32_t accumulate = 0;
#pragma unroll
              for (int dy = 0; dy < 3; ++dy) {
                const int sl = dy == 0 ? s_prev : (dy == 1 ? s_cur : s_next);
                if (sl >= 0) {
                  const uint32_t a_row = ring16 + (uint32_t)sl * row16 + simple_a;
#pragma unroll
                  for (int dx = 0; dx < 3; ++dx) {
                    umma_bf16(tmem_d, simple_hi | (a_row + (uint32_t)dx * simple_rowp), simple_hi | simple_w[dy * 3 + dx],
                              idesc, accumulate);
                    accumulate = 1;
                  }
                }
              }
            }
            __syncwarp();
          } else {
          uint32_t accumulate = 0;
#pragma unroll 1
            for (int dy = 0; dy < 3; ++dy) {
              const int sl = dy == 0 ? s_prev : (dy == 1 ? s_cur : s_next);
              if (sl < 0) continue;                    // zero padding row: contributes nothing
              const uint32_t a_row = ring16 + (uint32_t)sl * row16;
              const uint32_t w_tap = w16 + (uint32_t)(dy * 3) * tap16;
#pragma unroll 1
              for (int g = 0; g < nblk; ++g) {
                const uint4 bk = s_blk[g];             // {a offset, w offset, descriptor hi word, row pitch | k16 count << 16}
                const uint64_t hi = (uint64_t)bk.z << 32;
                const uint32_t rowp = bk.w & 0xFFFFu, nk16 = bk.w >> 16;
                if (elect_one()) {
#pragma unroll
                  for (int dx = 0; dx < 3; ++dx) {
                    // tap (dy, dx): rows [dx, dx + 128) of the halo'd row tile; weights of tap dy*3 + dx
                    const uint64_t adesc = hi | (a_row + bk.x + (uint32_t)dx * rowp);
                    const uint64_t bdesc = hi | (w_tap + (uint32_t)dx * tap16 + bk.y);
                    umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
                    accumulate = 1;
                    if (nk16 > 1) {
                      umma_bf16(tmem_d, adesc + 2, bdesc + 2, idesc, 1u);
                      if (nk16 > 2) {
                        umma_bf16(tmem_d, adesc + 4, bdesc + 4, idesc, 1u);
                        if (nk16 > 3) umma_bf16(tmem_d, adesc + 6, bdesc + 6, idesc, 1u);
                      }
                    }
                  }
                }
                accumulate = 1;
                __syncwarp();
              }
            }
          }
          if (elect_one()) {
            umma_commit(bar_tf0 + 8u * acc);
            // input row yo-1 has no later reader; the last output row of the unit also retires rows yo and yo+1
            if (s_prev >= 0) umma_commit(bar_empty0 + 8u * (uint32_t)s_prev);
            if (yo == y0 + R - 1) {
              umma_commit(bar_empty0 + 8u * (uint32_t)s_cur);
              if (s_next >= 0) umma_commit(bar_empty0 + 8u * (uint32_t)s_next);
            }
          }
          __syncwarp();
          s_prev = s_cur;
          s_cur = s_next;
        }
      }
    }
  } else {
    // ===================== epilogue: warps 2..5, warp w owns TMEM lanes 32*(w%4) .. +31 and all column chunks ==========
    // (NS > 0: a second group, warps 6..9, takes the odd accumulator stage)
    const int ew = warp & 3;
    const int grp = (warp - 2) >> 2;
    const int ewi = warp - 2;
    const int row = ew * 32 + lane;
    const int et = threadIdx.x - 64;
    epi_stage_vectors(p.e, s_bias, s_r1w, s_off, 0, p.block_n, et, EPI_GROUPS * RING_EPI_THREADS);
    int it = 0;
    for (int unit = blockIdx.x; unit < p.total_units; unit += gridDim.x) {
      const int rc = unit % p.chunks;
      const int xs = (unit / p.chunks) % p.strips;
      const int b = unit / (p.chunks * p.strips);
      const int y0 = rc * p.R, x0 = xs * TC_BM;
      for (int yo = y0; yo < y0 + p.R; ++yo, ++it) {
        const int acc = it & 1;
        if (EPI_GROUPS == 2 && acc != grp) continue;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        const int m_glob = (b * p.H + yo) * p.W + x0 + row;
        float rs = 1.f, r1 = 0.f;
        if (p.e.row_scale) rs = __ldg(p.e.row_scale + m_glob);
        if (p.e.row_r1) r1 = __ldg(p.e.row_r1 + m_glob);
        mbar_wait(smem_u32(&bar_tmem_full[acc]), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * p.block_n);
        if (STAGED) {
          epi_store_row_staged<MODE, HAS_R1>(p.e, taddr, 0, 1, p.block_n, 0, true, epi_row_base<MODE>(p.e, m_glob), rs, r1,
                                             s_bias, s_r1w, s_off, smem_u32(&bar_tmem_empty[acc]),
                                             s_stage + ewi * EPI_WARP_STAGE_BYTES, s_rowbase + 32 * ewi);
        } else {
          epi_store_row<MODE, HAS_R1, OUT_F32>(p.e, taddr, 0, p.block_n, 0, true, m_glob, epi_row_base<MODE>(p.e, m_glob),
                                               rs, r1, s_bias, s_r1w, s_off, 1, smem_u32(&bar_tmem_empty[acc]));
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------
static int round1k(int v) { return (v + 1023) / 1024 * 1024; }

static bool ring_stages_output(const ccvpe_igemm_desc& d) {
  return d.out_dtype == CCVPE_BF16 && d.out_mode != 2 && d.N >= 32;
}

static bool ring_plan(const ccvpe_igemm_desc& d, RingParams* p) {
  if (d.dtype != CCVPE_BF16 || !d.w_nk) return false;
  if (d.stride != 1 || d.kh != 3 || d.kw != 3 || d.pad != 1) return false;
  if (d.Hin != d.Hout || d.Win != d.Wout || d.Wout % TC_BM != 0) return false;
  if (d.out_mode == 1 || d.N > TC_MAX_N || d.relu == 2 || !tc_epilogue_supported(d)) return false;
  p->kw0 = tc_block_width(d.c0);
  p->kw1 = d.c1 ? tc_block_width(d.c1) : 64;
  p->nb0 = (d.c0 + p->kw0 - 1) / p->kw0;
  p->nb1 = d.c1 ? (d.c1 + p->kw1 - 1) / p->kw1 : 0;
  if (p->nb0 + p->nb1 > 4) return false;
  p->kpad0 = p->nb0 * p->kw0;
  p->kpad1 = p->nb1 * p->kw1;
  p->c0 = d.c0;
  p->c1 = d.c1;
  p->block_n = (d.N + 15) / 16 * 16;
  p->tmem_cols = 32;
  while (p->tmem_cols < 2 * p->block_n) p->tmem_cols <<= 1;
  p->a_blk0 = round1k(RING_HALO_W * p->kw0 * 2);
  p->a_blk1 = round1k(RING_HALO_W * p->kw1 * 2);
  p->row_bytes = p->nb0 * p->a_blk0 + p->nb1 * p->a_blk1;
  p->w_blk0 = round1k(p->block_n * p->kw0 * 2);
  p->w_blk1 = round1k(p->block_n * p->kw1 * 2);
  p->w_tap_bytes = p->nb0 * p->w_blk0 + p->nb1 * p->w_blk1;
  {
    int j = 0;
    uint32_t ao = 0, wo = 0;
    bool fits = true;
    for (int g = 0; g < p->nb0 + p->nb1 && fits; ++g) {
      const bool s1 = g >= p->nb0;
      const int kw = s1 ? p->kw1 : p->kw0, cb = s1 ? g - p->nb0 : g, c = s1 ? d.c1 : d.c0, nb = s1 ? p->nb1 : p->nb0;
      const int nk16 = (cb == nb - 1) ? (c - cb * kw + 15) / 16 : kw / 16;
      for (int k = 0; k < nk16; ++k, ++j) {
        if (j >= RING_MAX_STEPS) {
          fits = false;
          break;
        }
        p->st_hi[j] = (uint32_t)(make_smem_desc(0, kw) >> 32);
        for (int dx = 0; dx < 3; ++dx) p->st_adx[j][dx] = ((ao + 32u * k) >> 4) + (uint32_t)dx * ((uint32_t)(kw * 2) >> 4);
        for (int t = 0; t < 9; ++t) p->st_wt[t][j] = ((uint32_t)t * (uint32_t)p->w_tap_bytes + wo + 32u * k) >> 4;
      }
      ao += s1 ? p->a_blk1 : p->a_blk0;
      wo += s1 ? p->w_blk1 : p->w_blk0;
    }
    p->n_steps = fits ? j : 0;
    // the plain bf16 channels-last convs with 2..4 K16 slices per tap (levels 2 and 3) take the unrolled issue path
    const bool plain = d.relu != 2 && d.out_mode == 0 && d.out_dtype == CCVPE_BF16 && !d.row_r1;            // epilogue variant 0
    p->unrolled = (plain && ring_stages_output(d) && p->n_steps >= 2 && p->n_steps <= 4) ? 1 : 0;
  }
  p->tx_row = (p->nb0 * p->kw0 + p->nb1 * p->kw1) * RING_HALO_W * 2;
  p->tx_weights = 9 * (p->nb0 * p->kw0 + p->nb1 * p->kw1) * p->block_n * 2;
  // (the second epilogue group's staging tiles are static shared memory: 11 KB less for the ring)
  const int avail = RING_SMEM_BUDGET - (p->unrolled ? 12 * 1024 : 0) - 9 * p->w_tap_bytes;
  if (avail < 4 * p->row_bytes) return false;
  int depth = avail / p->row_bytes;
  p->depth = depth > RING_MAX_DEPTH ? RING_MAX_DEPTH : depth;
  // prefer a shallower ring if that lets two CTAs (two MMA issuers, two producers, eight epilogue warps) share an SM:
  // the narrow levels are bound by single-thread issue latency, not by pipeline depth
  // static shared memory + alignment slack of one CTA (the bf16 variants carry the epilogue staging tiles)
  // (the unrolled variants: two epilogue groups -> twice the staging tiles, 320 threads -> at most two CTAs per SM)
  const int static_bytes = p->unrolled ? 28 * 1024 : (ring_stages_output(d) ? 15 * 1024 : 4096);
  bool placed = false;
  for (int ctas = p->unrolled ? 2 : 3; ctas >= 2 && !placed; --ctas) {
    for (int dd = p->depth; dd >= 4; --dd) {
      if (ctas * (9 * p->w_tap_bytes + dd * p->row_bytes + static_bytes) <= 224 * 1024) {
        p->depth = dd;
        placed = true;
        break;
      }
    }
  }
  p->B = d.B;
  p->H = d.Hout;
  p->W = d.Wout;
  p->strips = d.Wout / TC_BM;
  int R = 32;
  while (R > 4 && ((int64_t)d.B * p->strips * (d.Hout / R) < 3 * (int64_t)sm_count() || d.Hout % R != 0)) R >>= 1;
  if (d.Hout % R != 0) return false;
  p->R = R;
  p->chunks = d.Hout / R;
  p->total_units = d.B * p->strips * p->chunks;
  return true;
}

bool conv_ring_supported(const ccvpe_igemm_desc& d) {
  static thread_local RingParams probe;
  return ring_plan(d, &probe);
}

int conv_ring_tcgen05(const ccvpe_igemm_desc& d, cudaStream_t st) {
  static thread_local RingParams p;
  memset(&p, 0, sizeof(p));
  if (!ring_plan(d, &p)) return fail(CCVPE_ERR_UNSUPPORTED, "conv_ring_tcgen05: unsupported shape");
  int rc;
  const uint64_t esz = 2;
  for (int s = 0; s < (d.c1 ? 2 : 1); ++s) {
    const void* base = s ? d.a1 : d.a0;
    const int c = s ? d.c1 : d.c0, ld = s ? d.ld1 : d.ld0, kw = s ? p.kw1 : p.kw0;
    uint64_t dims[3] = {(uint64_t)c, (uint64_t)d.Win, (uint64_t)d.B * d.Hin};
    uint64_t str[2] = {(uint64_t)ld * esz, (uint64_t)d.Win * ld * esz};
    uint32_t box[3] = {(uint32_t)kw, (uint32_t)RING_HALO_W, 1};
    if ((rc = encode_map(s ? &p.tm_a1 : &p.tm_a0, base, 3, dims, str, box, kw)) != CCVPE_OK) return rc;
    const uint64_t ktot = 9ull * (p.kpad0 + p.kpad1);
    uint64_t wdims[2] = {ktot, (uint64_t)d.N};
    uint64_t wstr[1] = {ktot * esz};
    uint32_t wbox[2] = {(uint32_t)kw, (uint32_t)p.block_n};
    if ((rc = encode_map(s ? &p.tm_b1 : &p.tm_b0, d.w_nk, 2, wdims, wstr, wbox, kw)) != CCVPE_OK) return rc;
  }
  fill_epi(p.e, d);
  const int smem = 9 * p.w_tap_bytes + p.depth * p.row_bytes + 1024;
  int ctas_per_sm = (224 * 1024) / (smem + (p.unrolled ? 26 * 1024 : 3072));   // shared memory (+ static) ...
  if (ctas_per_sm > 512 / p.tmem_cols) ctas_per_sm = 512 / p.tmem_cols;   // ... TMEM columns ...
  if (ctas_per_sm > (p.unrolled ? 2 : 3)) ctas_per_sm = p.unrolled ? 2 : 3;   // ... registers / threads (launch bounds)
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  const int max_grid = ctas_per_sm * sm_count();
  const int grid = p.total_units < max_grid ? p.total_units : max_grid;
  cudaError_t attr_err = cudaSuccess;
#define CCVPE_LAUNCH_RING(MODE, R1, F32)                                                                         \
  do {                                                                                                           \
    static thread_local uint64_t attr = 0;                                                                       \
    if (first_use_on_device(attr)) {                                                                             \
      attr_err = cudaFuncSetAttribute(conv_ring_tcgen05_kernel<MODE, R1, F32, false>,                            \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, RING_SMEM_BUDGET + 2048);     \
      if (!(F32) && MODE != 2 && attr_err == cudaSuccess)                                                        \
        attr_err = cudaFuncSetAttribute(conv_ring_tcgen05_kernel<MODE, R1, F32, !(F32) && MODE != 2>,            \
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, RING_SMEM_BUDGET + 2048);   \
    }                                                                                                            \
    if (stage_out) conv_ring_tcgen05_kernel<MODE, R1, F32, !(F32) && MODE != 2><<<grid, RING_THREADS, smem, st>>>(p); \
    else conv_ring_tcgen05_kernel<MODE, R1, F32, false><<<grid, RING_THREADS, smem, st>>>(p);                     \
  } while (0)
#define CCVPE_LAUNCH_RING_NS(NSV)                                                                                \
  do {                                                                                                           \
    static thread_local uint64_t attr = 0;                                                                       \
    if (first_use_on_device(attr))                                                                               \
      attr_err = cudaFuncSetAttribute(conv_ring_tcgen05_kernel<0, false, false, true, NSV>,                      \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, RING_SMEM_BUDGET - 10 * 1024); \
    conv_ring_tcgen05_kernel<0, false, false, true, NSV><<<grid, RING_THREADS + RING_EPI_THREADS, smem, st>>>(p); \
  } while (0)
  const bool stage_out = ring_stages_output(d);
  if (p.unrolled) {
    if (p.n_steps == 2) CCVPE_LAUNCH_RING_NS(2);
    else if (p.n_steps == 3) CCVPE_LAUNCH_RING_NS(3);
    else CCVPE_LAUNCH_RING_NS(4);
  } else {
    CCVPE_EPI_SWITCH(epi_variant(p.e), CCVPE_LAUNCH_RING)
  }
#undef CCVPE_LAUNCH_RING_NS
#undef CCVPE_LAUNCH_RING
  if (attr_err != cudaSuccess) return fail(CCVPE_ERR_CUDA, "cudaFuncSetAttribute(ring): %s", cudaGetErrorString(attr_err));
  return check_launch("conv_ring_tcgen05_kernel");
}

}  // namespace ccvpe
