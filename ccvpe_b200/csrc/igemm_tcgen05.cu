// tcgen05 backend of the generic implicit GEMM: the bf16 throughput path of a3 (cell descriptors), a8 (transposed
// convs) and a9 (3x3 convs).  sm_100a only.
//
//   * A (activations, channels-last bf16) is never im2col'ed: for every (tap, 64-channel block) ONE TMA box load of
//     [128 pixels x 64 channels] at spatially shifted coordinates lands a K-major, 128B-swizzled UMMA operand tile in
//     shared memory; the conv halo (pad 1) is TMA out-of-bounds zero fill, channel tails are zero filled too, and the
//     skip concat is a second tensor map walked by the same K loop.
//   * B (weights, [N][taps][K] bf16, K contiguous) tiles arrive through a 2-D tensor map the same way.
//   * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=block_n<=256, K=16) into TMEM; accumulators
//     are double buffered (2 x 256 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
//   * warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..7 = epilogue (tcgen05.ld -> bias / row-scale /
//     rank-1 / ReLU -> bf16 or fp32 stores incl. the transposed-conv pixel shuffle).  Persistent: grid = min(tiles, SMs).
//   * every mbarrier wait is bounded (clock64 watchdog -> __trap) so a protocol bug fails the launch instead of
//     hanging the GPU.
#include "tcgen05_common.cuh"

namespace ccvpe {

// warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner, warps 2..9 = epilogue.  Two instantiations: HEAVY (one CTA per
// SM, all of its shared memory as pipeline stages: wide compute-bound tiles) and LIGHT (two CTAs share an SM: two
// producers / MMA issuers and 16 epilogue warps for the narrow HBM-bound layers, which are limited by single-thread issue
// and by the epilogue's instruction latencies; its rows leave through shared-memory staging tiles).
constexpr int TC_MAX_STAGES = 16;
constexpr int TC_SMEM_BUDGET = 200 * 1024;

struct TcParams {
  CUtensorMap tm_a0, tm_a1, tm_b0, tm_b1;
  int nb0, nb1, c0, c1, kw0, kw1, kpad0, kpad1, taps, n_tiles_n, total_tiles, block_n, stages, a_bytes, stage_bytes;
  int tmem_cols, a_rank;      // a_rank: rank of the A tensor maps (2 = flattened pixels, 4 = [C,W,H,B], 5 = cell gather)
  int tiles[4], box[4];
  int tile_shift[4], box_shift[4];   // tiles[] / box[] are powers of two (the last non-unit tiles[] entry takes "the rest")
  int tap_off[9][4];
  int out_stride[4], extent[4];
  int pad_w, pad_h, pad_wp, pad_hp, pad_lo;   // MODE 3 only: rows are written into the interior of a padded image
  int epi_off;                                // byte offset of the epilogue staging tile behind the pipeline stages
  int w_resident, w_off, w_blk;               // weights loaded once per CTA: offset of / bytes per K-block B tile
  // halo mode (3x3 convs of the shallow levels): ONE A box [(th+2) x (tw+2) px x kw ch] per K block serves all nine taps
  // (tile = 8 x 16 pixels, so a UMMA 8-row group is one image row and the group stride is the halo pitch); the nine
  // weight tiles stream through the ordinary stage ring
  int halo, a_slots, a_slot_bytes, b_off, halo_pitch, halo_tx0, halo_tx1;
  EpiParams e;
};

constexpr int TC_HALO_SLOTS = 4;

// ---- kernel ------------------------------------------------------------------------------------------------------
template <bool LIGHT, int MODE, bool HAS_R1, bool OUT_F32>
__global__ void __launch_bounds__(64 + 32 * TC_EPI_WARPS, LIGHT ? 2 : 1)
igemm_tcgen05_kernel(const __grid_constant__ TcParams p) {
  constexpr int EPI_WARPS = TC_EPI_WARPS;
  constexpr int EPI_THREADS = 32 * EPI_WARPS;
  // the light (two CTAs per SM) configuration runs the HBM-bound layers: its bf16 rows leave through per-warp staging tiles
  constexpr bool STAGED = LIGHT && !OUT_F32 && MODE != 2;
  extern __shared__ uint8_t smem_raw[];
  __shared__ int32_t s_rowbase[STAGED ? 32 * EPI_WARPS : 1];
  __shared__ __align__(8) uint64_t bar_full[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_empty[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full[2];
  __shared__ __align__(8) uint64_t bar_tmem_empty[2];
  __shared__ __align__(8) uint64_t bar_weights;
  __shared__ __align__(8) uint64_t bar_a_full[TC_HALO_SLOTS];
  __shared__ __align__(8) uint64_t bar_a_empty[TC_HALO_SLOTS];
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float s_bias[2][TC_MAX_N];
  __shared__ __align__(16) float s_r1w[2][TC_MAX_N];
  __shared__ int s_off[2][TC_MAX_N / 8];

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int stage_bytes = p.stage_bytes;   // A tile + B tile of the widest K block in use, 1024-byte aligned
  const int nkb = p.taps * (p.nb0 + p.nb1);

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tmem_full[a]), 1);
      mbar_init(smem_u32(&bar_tmem_empty[a]), EPI_WARPS);
    }
    mbar_init(smem_u32(&bar_weights), 1);
    for (int s2 = 0; s2 < TC_HALO_SLOTS; ++s2) {
      mbar_init(smem_u32(&bar_a_full[s2]), 1);
      mbar_init(smem_u32(&bar_a_empty[s2]), 1);
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
  // Tile schedule.  Streaming mode: CTA c takes tiles c, c + grid, ... of the (m tile, n tile) grid, n fastest.  Resident
  // mode (weights of ONE N tile stay in shared memory): CTA c owns N tile c % n_tiles_n and walks the m tiles
  // c / n_tiles_n, + grid / n_tiles_n, ...  Either way `tile` below runs t0, t0 + tstep, ... < tend.
  const bool res = p.w_resident != 0;
  const int cta_nt = res ? (int)blockIdx.x % p.n_tiles_n : 0;
  const int t0 = res ? (int)blockIdx.x / p.n_tiles_n : (int)blockIdx.x;
  const int tstep = res ? (int)gridDim.x / p.n_tiles_n : (int)gridDim.x;
  const int tend = res ? p.total_tiles / p.n_tiles_n : p.total_tiles;
  const bool fixed_n = res || p.n_tiles_n == 1;     // the N tile never changes within this CTA

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged, single-lane issue via elect_one) =====================
    {
      if (res && t0 < tend) {
        // this CTA's N tile of the weight matrix stays in shared memory: one K-block B tile per (tap, source, block).
        // Re-fetching it per tile would make every CTA hammer the same few L2 lines all the time.
        if (elect_one()) {
          const uint32_t bw = smem_u32(&bar_weights);
          uint32_t bytes = 0;
          for (int tap = 0; tap < p.taps; ++tap)
            bytes += (uint32_t)(p.block_n * 2 * (p.nb0 * p.kw0 + p.nb1 * p.kw1));
          mbar_arrive_expect_tx(bw, bytes);
          int kb = 0;
          for (int tap = 0; tap < p.taps; ++tap)
            for (int src = 0; src < 2; ++src) {
              const int nb = src ? p.nb1 : p.nb0, kw = src ? p.kw1 : p.kw0;
              const int kbase = tap * (p.kpad0 + p.kpad1) + (src ? p.kpad0 : 0);
              for (int cb = 0; cb < nb; ++cb, ++kb)
                tma_load_2d(smem_base + p.w_off + kb * p.w_blk, src ? &p.tm_b1 : &p.tm_b0, bw, kbase + cb * kw,
                            cta_nt * p.block_n);
            }
        }
        __syncwarp();
      }
      int stage = 0;
      uint32_t phase = 0;
      int aslot = 0;
      uint32_t aphase = 0;
      for (int tile = t0; tile < tend; tile += tstep) {
        int mt = fixed_n ? tile : tile / p.n_tiles_n;
        const int nt = fixed_n ? cta_nt : tile - mt * p.n_tiles_n;
        int base[4];
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          base[d] = (mt & ((1 << p.tile_shift[d]) - 1)) << p.box_shift[d];
          mt >>= p.tile_shift[d];
        }
        const int n0 = nt * p.block_n;
        if (p.halo) {
          // per K block: one halo box of the activations, then the nine tap tiles of the weights
          for (int src = 0; src < 2; ++src) {
            const int nb = src ? p.nb1 : p.nb0;
            const int kw = src ? p.kw1 : p.kw0;
            const CUtensorMap* tm = src ? &p.tm_a1 : &p.tm_a0;
            const CUtensorMap* tmb = src ? &p.tm_b1 : &p.tm_b0;
            const uint32_t txb = (uint32_t)(p.block_n * kw * 2);
            for (int cb = 0; cb < nb; ++cb) {
              mbar_wait(smem_u32(&bar_a_empty[aslot]), aphase ^ 1u);
              if (elect_one()) {
                const uint32_t full = smem_u32(&bar_a_full[aslot]);
                mbar_arrive_expect_tx(full, (uint32_t)(src ? p.halo_tx1 : p.halo_tx0));
                tma_load_4d(smem_base + aslot * p.a_slot_bytes, tm, full, cb * kw, base[0] - 1, base[1] - 1, base[2]);
              }
              __syncwarp();
              if (++aslot == p.a_slots) {
                aslot = 0;
                aphase ^= 1u;
              }
              for (int tap = 0; tap < 9; ++tap) {
                const int kbase = tap * (p.kpad0 + p.kpad1) + (src ? p.kpad0 : 0);
                mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
                if (elect_one()) {
                  const uint32_t full = smem_u32(&bar_full[stage]);
                  mbar_arrive_expect_tx(full, txb);
                  tma_load_2d(smem_base + p.b_off + stage * stage_bytes, tmb, full, kbase + cb * kw, n0);
                }
                __syncwarp();
                if (++stage == p.stages) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
          }
          continue;
        }
        for (int tap = 0; tap < p.taps; ++tap) {
          const int c1 = base[0] + p.tap_off[tap][0], c2 = base[1] + p.tap_off[tap][1];
          const int c3 = base[2] + p.tap_off[tap][2], c4 = base[3] + p.tap_off[tap][3];
          for (int src = 0; src < 2; ++src) {
            const int nb = src ? p.nb1 : p.nb0;
            const int kw = src ? p.kw1 : p.kw0;
            const CUtensorMap* tm = src ? &p.tm_a1 : &p.tm_a0;
            const CUtensorMap* tmb = src ? &p.tm_b1 : &p.tm_b0;
            const int kbase = tap * (p.kpad0 + p.kpad1) + (src ? p.kpad0 : 0);   // column of this source in W[n][.]
            const uint32_t tx = (uint32_t)((TC_BM + (p.w_resident ? 0 : p.block_n)) * kw * 2);
            for (int cb = 0; cb < nb; ++cb) {
              mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
              if (elect_one()) {
                const uint32_t full = smem_u32(&bar_full[stage]);
                const uint32_t a_dst = smem_base + stage * stage_bytes;
                mbar_arrive_expect_tx(full, tx);
                // lowest-rank map that expresses the access: TMA issue cost grows with rank (scripts/tma_probe.cu)
                if (p.a_rank == 2) tma_load_2d(a_dst, tm, full, cb * kw, c1);
                else if (p.a_rank == 4) tma_load_4d(a_dst, tm, full, cb * kw, c1, c2, c3);
                else tma_load_5d(a_dst, tm, full, cb * kw, c1, c2, c3, c4);
                if (!p.w_resident) tma_load_2d(a_dst + p.a_bytes, tmb, full, kbase + cb * kw, n0);
              }
              __syncwarp();
              if (++stage == p.stages) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // One thread issues everything, so the per-K-block instruction count is the pipeline's clock: all descriptor
    // pieces are precomputed and the loop nest mirrors the producer's (no div/mod in the steady state).  The warp stays
    // converged; the MMAs and commits are predicated with elect_one().
    {
      // instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=block_n
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.block_n >> 3) << 17) |
                             ((uint32_t)(TC_BM >> 4) << 24);
      const uint32_t hi0 = (uint32_t)(make_smem_desc(0, p.kw0) >> 32), hi1 = (uint32_t)(make_smem_desc(0, p.kw1) >> 32);
      const int full0 = p.kw0 >> 4, full1 = p.kw1 >> 4;
      const int tail0 = (p.c0 - (p.nb0 - 1) * p.kw0 + 15) >> 4, tail1 = p.nb1 ? (p.c1 - (p.nb1 - 1) * p.kw1 + 15) >> 4 : 0;
      const uint32_t lo_base = ((smem_base & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t lo_stage = (uint32_t)stage_bytes >> 4, lo_b = (uint32_t)p.a_bytes >> 4;
      const uint32_t lo_w = ((((smem_base + (uint32_t)p.w_off) & 0x3FFFFu) >> 4) | (1u << 16)), lo_wblk = (uint32_t)p.w_blk >> 4;
      if (res && t0 < tend) {
        mbar_wait(smem_u32(&bar_weights), 0);
        tc_fence_after();
      }
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      int aslot = 0;
      uint32_t aphase = 0;
      // halo mode: A descriptors address the halo tile (group stride = halo pitch), B descriptors the weight ring
      const uint32_t lo_bring = ((((smem_base + (uint32_t)p.b_off) & 0x3FFFFu) >> 4) | (1u << 16));
      const uint32_t lo_aslot = (uint32_t)p.a_slot_bytes >> 4;
      for (int tile = t0; tile < tend; tile += tstep, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(smem_u32(&bar_tmem_empty[acc]), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * p.block_n);
        uint32_t accumulate = 0;
        uint32_t b_res = lo_w;                     // resident B tile of the next K block
        if (p.halo) {
#pragma unroll 1
          for (int src = 0; src < 2; ++src) {
            const int nb = src ? p.nb1 : p.nb0;
            const int kw = src ? p.kw1 : p.kw0;
            const uint32_t hib = src ? hi1 : hi0;
            const uint32_t row_units = (uint32_t)(kw * 2) >> 4;                       // one pixel of the halo tile
            const uint32_t hia = (hib & ~0x3FFFu) | ((uint32_t)p.halo_pitch * row_units);   // SBO = one halo row of pixels
            const uint32_t pitch_units = (uint32_t)p.halo_pitch * row_units;
            const int nfull = src ? full1 : full0, ntail = src ? tail1 : tail0;
#pragma unroll 1
            for (int cb = 0; cb < nb; ++cb) {
              const int nk16 = (cb == nb - 1) ? ntail : nfull;
              mbar_wait(smem_u32(&bar_a_full[aslot]), aphase);
              tc_fence_after();
              const uint32_t a_lo0 = lo_base + (uint32_t)aslot * lo_aslot;
#pragma unroll
              for (int tap = 0; tap < 9; ++tap) {
                mbar_wait(smem_u32(&bar_full[stage]), phase);
                tc_fence_after();
                const uint64_t adesc = ((uint64_t)hia << 32) | (a_lo0 + (uint32_t)(tap / 3) * pitch_units + (uint32_t)(tap % 3) * row_units);
                const uint64_t bdesc = ((uint64_t)hib << 32) | (lo_bring + (uint32_t)stage * lo_stage);
                if (elect_one()) {
                  umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
                  if (nk16 > 1) umma_bf16(tmem_d, adesc + 2, bdesc + 2, idesc, 1u);
                  if (nk16 > 2) umma_bf16(tmem_d, adesc + 4, bdesc + 4, idesc, 1u);
                  if (nk16 > 3) umma_bf16(tmem_d, adesc + 6, bdesc + 6, idesc, 1u);
                  umma_commit(smem_u32(&bar_empty[stage]));
                  if (tap == 8) umma_commit(smem_u32(&bar_a_empty[aslot]));          // the halo tile is free again
                }
                accumulate = 1;
                __syncwarp();
                if (++stage == p.stages) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
              if (++aslot == p.a_slots) {
                aslot = 0;
                aphase ^= 1u;
              }
            }
          }
          if (elect_one()) umma_commit(smem_u32(&bar_tmem_full[acc]));
          __syncwarp();
          continue;
        }
        for (int tap = 0; tap < p.taps; ++tap) {
#pragma unroll 1
          for (int src = 0; src < 2; ++src) {
            const int nb = src ? p.nb1 : p.nb0;
            const uint32_t hi = src ? hi1 : hi0;
            const int nfull = src ? full1 : full0, ntail = src ? tail1 : tail0;
#pragma unroll 1
            for (int cb = 0; cb < nb; ++cb) {
              const int nk16 = (cb == nb - 1) ? ntail : nfull;
              mbar_wait(smem_u32(&bar_full[stage]), phase);
              tc_fence_after();
              const uint32_t a_lo = lo_base + (uint32_t)stage * lo_stage;
              const uint64_t adesc = ((uint64_t)hi << 32) | a_lo;
              const uint64_t bdesc = ((uint64_t)hi << 32) | (p.w_resident ? b_res : a_lo + lo_b);
              b_res += lo_wblk;
              if (elect_one()) {
                // k-th MMA: advance 16 bf16 = 32 bytes inside the swizzle row (+2 in the 16-byte address field)
                umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
                if (nk16 > 1) umma_bf16(tmem_d, adesc + 2, bdesc + 2, idesc, 1u);
                if (nk16 > 2) umma_bf16(tmem_d, adesc + 4, bdesc + 4, idesc, 1u);
                if (nk16 > 3) umma_bf16(tmem_d, adesc + 6, bdesc + 6, idesc, 1u);
                umma_commit(smem_u32(&bar_empty[stage]));   // frees the smem slot once these MMAs have read it
              }
              accumulate = 1;
              __syncwarp();
              if (++stage == p.stages) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
        }
        if (elect_one()) umma_commit(smem_u32(&bar_tmem_full[acc]));    // accumulator complete -> epilogue
        __syncwarp();
      }
    }
  } else {
    // ===== epilogue: 8 warps; warp w reads TMEM lanes 32*(w%4) .. +31 and every other 32-column chunk ((w-4)/4) =====
    const int ew = warp & 3;
    const int half = (warp - 2) >> 2;                 // which interleaved set of 32-column chunks
    const int row = ew * 32 + lane;
    const int et = threadIdx.x - 64;                  // index within the epilogue group
    const bool has_r1 = (p.e.row_r1 != nullptr), has_rs = (p.e.row_scale != nullptr);
    // row -> output pixel of a tile
    // (shifts and masks only: this runs per tile in every epilogue thread)
    auto locate = [&](int tile, int& m_glob, bool& valid, int64_t& row_base) {
      int mt = fixed_n ? tile : tile / p.n_tiles_n;
      if (p.a_rank == 2) {
        m_glob = mt * TC_BM + row;
        valid = m_glob < p.extent[0];
      } else {
        int r = row;
        m_glob = 0;
        valid = true;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          const int coord = ((mt & ((1 << p.tile_shift[d]) - 1)) << p.box_shift[d]) + (r & ((1 << p.box_shift[d]) - 1));
          mt >>= p.tile_shift[d];
          r >>= p.box_shift[d];
          valid = valid && (coord < p.extent[d]);
          m_glob += coord * p.out_stride[d];
        }
      }
      int m_out = m_glob;
      if (MODE == 3 && p.pad_w) {   // (b, h, w) -> interior pixel of the padded [B, Hp, Wp] staging image
        const int q = m_glob / p.pad_w, w = m_glob - q * p.pad_w;
        const int b = q / p.pad_h, h = q - b * p.pad_h;
        m_out = (b * p.pad_hp + h + p.pad_lo) * p.pad_wp + w + p.pad_lo;
      }
      row_base = epi_row_base<MODE>(p.e, m_out);
    };

    if (fixed_n) epi_stage_vectors(p.e, s_bias[0], s_r1w[0], s_off[0], cta_nt * p.block_n, p.block_n, et, EPI_THREADS);
    int m_glob, m_next = 0;
    int64_t row_base, base_next = 0;
    bool valid, valid_next = false;
    float rs = 1.f, r1 = 0.f, rs_next = 1.f, r1_next = 0.f;
    if (t0 < tend) {
      locate(t0, m_next, valid_next, base_next);
      if (valid_next) {
        if (has_rs) rs_next = __ldg(p.e.row_scale + m_next);
        if (has_r1) r1_next = __ldg(p.e.row_r1 + m_next);
      }
    }
    int it = 0;
    for (int tile = t0; tile < tend; tile += tstep, ++it) {
      m_glob = m_next; valid = valid_next; rs = rs_next; r1 = r1_next; row_base = base_next;
      {  // prefetch the per-row scalars of the next tile: their latency hides behind this tile's epilogue
        const int nxt = tile + tstep;
        rs_next = 1.f; r1_next = 0.f; valid_next = false;
        if (nxt < tend) {
          locate(nxt, m_next, valid_next, base_next);
          if (valid_next) {
            if (has_rs) rs_next = __ldg(p.e.row_scale + m_next);
            if (has_r1) r1_next = __ldg(p.e.row_r1 + m_next);
          }
        }
      }
      const int n0 = (fixed_n ? cta_nt : tile % p.n_tiles_n) * p.block_n;
      const int acc = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      const int vb = fixed_n ? 0 : acc;
      if (!fixed_n) epi_stage_vectors(p.e, s_bias[acc], s_r1w[acc], s_off[acc], n0, p.block_n, et, EPI_THREADS);
      mbar_wait(smem_u32(&bar_tmem_full[acc]), acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * p.block_n);
      // (the accumulator stage is released to the MMA issuer inside, once its last chunk has been read)
      if (STAGED) {
        const int ewi = warp - 2;                     // index among the epilogue warps
        epi_store_row_staged<MODE, HAS_R1>(p.e, taddr, half, EPI_WARPS / 4, p.block_n, n0, valid, row_base, rs, r1,
                                           s_bias[vb], s_r1w[vb], s_off[vb], smem_u32(&bar_tmem_empty[acc]),
                                           smem_raw + (smem_base - smem_u32(smem_raw)) + p.epi_off +
                                               ewi * EPI_WARP_STAGE_BYTES,
                                           s_rowbase + 32 * ewi);
      } else {
        epi_store_row<MODE, HAS_R1, OUT_F32>(p.e, taddr, half, p.block_n, n0, valid, m_glob, row_base, rs, r1, s_bias[vb],
                                             s_r1w[vb], s_off[vb], EPI_WARPS / 4, smem_u32(&bar_tmem_empty[acc]));
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

static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

struct TcGeometry {
  bool cell;        // k2 s2 gather (aerial cell descriptors; data gradient of the k2 s2 transposed convs)
  bool halo;        // 3x3 conv with one halo A box per K block (8 x 16 pixel tiles)
  int tw, th, tb;   // conv tile: tw x th pixels x tb images = 128 rows (cell: tw output columns x th (row, image) pairs)
};

static bool tc_geometry(const ccvpe_igemm_desc& d, TcGeometry* g) {
  if (d.stride == 2 && d.kh == 2 && d.kw == 2 && d.pad == 0) {
    if (d.Hin != 2 * d.Hout || d.Win != 2 * d.Wout || d.c1 != 0 || !is_pow2(d.Wout)) return false;
    g->cell = true;
    g->halo = false;
    g->tw = d.Wout < TC_BM ? d.Wout : TC_BM;
    g->th = TC_BM / g->tw;
    g->tb = 0;
    return true;
  }
  if (d.stride != 1 || d.kh != d.kw || !(d.kh == 1 || d.kh == 3) || d.pad != (d.kh - 1) / 2) return false;
  if (d.Hin != d.Hout || d.Win != d.Wout) return false;
  if (d.kh == 1) {   // 1x1: flattened pixel tiles, any spatial size
    g->cell = false;
    g->halo = false;
    g->tw = TC_BM;
    g->th = g->tb = 1;
    return true;
  }
  if (!is_pow2(d.Wout) || !is_pow2(d.Hout)) return false;
  g->halo = false;
  // one halo A box per K block for the shallow 3x3 layers (N <= 160), which are bound by TMA's per-box-row issue rate
  // when every tap loads its own 128-row A box (9 x 128 rows per K block vs 180 for the halo box)
  if (d.Wout >= 8 && d.Hout >= 16 && d.N <= 160) {
    g->cell = false;
    g->halo = true;
    g->tw = 8;
    g->th = 16;
    g->tb = 1;
    return true;
  }
  int tw = d.Wout < TC_BM ? d.Wout : TC_BM;
  int th = TC_BM / tw;
  if (th > d.Hout) th = d.Hout;
  int tb = TC_BM / (tw * th);
  if (tw * th * tb != TC_BM || tb > 256) return false;
  g->cell = false;
  g->tw = tw;
  g->th = th;
  g->tb = tb;
  return true;
}

bool igemm_tcgen05_supported(const ccvpe_igemm_desc& d) {
  TcGeometry g;
  if (d.dtype != CCVPE_BF16 || !d.w_nk) return false;
  if (!tc_geometry(d, &g)) return false;
  if (d.out_mode == 1 && (d.kh != 1)) return false;
  if (!tc_epilogue_supported(d)) return false;
  return true;
}

static int ilog2(int v) {
  int s = 0;
  while ((1 << s) < v) ++s;
  return s;
}

int igemm_tcgen05(const ccvpe_igemm_desc& d, cudaStream_t st, const TcOutPad* out_pad) {
  TcGeometry g;
  if (d.dtype != CCVPE_BF16) return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): bf16 operands only");
  if (!d.w_nk) return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_igemm(tcgen05): w_nk is null");
  if (!tc_geometry(d, &g)) return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): unsupported geometry");
  if (!aligned16(d.w_nk)) return fail(CCVPE_ERR_BAD_ARGUMENT, "ccvpe_igemm(tcgen05): w_nk must be 16-byte aligned");
  if (!tc_epilogue_supported(d))
    return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): bf16 outputs need channel counts / ldo that are multiples "
                                       "of 8 and a 16-byte aligned base");
  if (d.relu == 2 && (d.out_mode != 0 || d.out_dtype != CCVPE_BF16 || d.row_r1))
    return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): SiLU epilogue is channels-last bf16 only");

  static thread_local TcParams p;   // > 1 KB: keep it off the stack; it is copied at launch
  memset(&p, 0, sizeof(p));
  p.kw0 = tc_block_width(d.c0);
  p.kw1 = d.c1 ? tc_block_width(d.c1) : 64;
  p.nb0 = (d.c0 + p.kw0 - 1) / p.kw0;
  p.nb1 = (d.c1 + p.kw1 - 1) / p.kw1;
  p.kpad0 = p.nb0 * p.kw0;
  p.kpad1 = p.nb1 * p.kw1;
  p.c0 = d.c0;
  p.c1 = d.c1;
  p.taps = d.kh * d.kw;
  // shallow-K layers are HBM / issue bound, not tensor bound: their tiles stay <= 128 columns so that two CTAs (two
  // producers / MMA issuers, 16 epilogue warps) fit an SM -- the LIGHT configuration, whose bf16 rows leave through the
  // per-warp staging tiles; everything else gets one HEAVY CTA per SM with all of its shared memory as pipeline stages.
  const int kw_max = (d.c1 && p.kw1 > p.kw0) ? p.kw1 : p.kw0;
  p.a_bytes = TC_BM * kw_max * 2;                                   // multiple of 1024 for every kw
  const bool shallow = p.taps * (d.c0 + d.c1) <= 256;
  const bool staged_out = d.out_dtype == CCVPE_BF16 && d.out_mode != 2;
  const int light_budget = 104 * 1024 - (staged_out ? TC_EPI_WARPS * EPI_WARP_STAGE_BYTES : 0);
  int n_tiles_n = 0, block_n = 0, stage_bytes = 0, w_bytes = 0;
  const int nkb_total = p.taps * (p.nb0 + p.nb1);
  auto plan = [&](int max_n) {
    n_tiles_n = (d.N + max_n - 1) / max_n;
    block_n = ((d.N + n_tiles_n - 1) / n_tiles_n + 15) / 16 * 16;
    const int b_blk = (block_n * kw_max * 2 + 1023) / 1024 * 1024;           // B tile of the widest K block in use
    p.tmem_cols = 32;
    while (p.tmem_cols < 2 * block_n) p.tmem_cols <<= 1;
    // an N tile whose weights fit next to >= 4 A stages stays resident in its CTAs (loaded once per CTA)
    p.w_resident = (p.tmem_cols <= 256 && nkb_total * b_blk <= 48 * 1024 &&
                    (light_budget - nkb_total * b_blk) / p.a_bytes >= 4) ? 1 : 0;
    p.w_blk = b_blk;
    w_bytes = p.w_resident ? nkb_total * b_blk : 0;
    stage_bytes = p.a_bytes + (p.w_resident ? 0 : b_blk);
    return p.tmem_cols <= 256 && (light_budget - w_bytes) / stage_bytes >= 3;
  };
  bool light = plan(shallow ? 128 : TC_MAX_N);
  if (!light && shallow) {            // wide K blocks: narrower N tiles keep three pipeline stages within the light budget
    light = plan(64);
    if (!light) plan(128);
  }
  p.n_tiles_n = n_tiles_n;
  p.block_n = block_n;
  p.stage_bytes = stage_bytes;
  if (!light && p.w_resident) {   // (cannot happen with the thresholds above; keep the two modes consistent anyway)
    p.w_resident = 0;
    w_bytes = 0;
    stage_bytes = p.a_bytes + p.w_blk;
  }
  int stages = (light ? light_budget - w_bytes : TC_SMEM_BUDGET) / stage_bytes;
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (g.halo) {
    // a ring of halo A tiles + a ring of weight tiles (weights stream: nine tiles per K block).
    p.w_resident = 0;
    w_bytes = 0;
    p.halo = 1;
    p.halo_pitch = g.tw + 2;
    p.halo_tx0 = (g.tw + 2) * (g.th + 2) * p.kw0 * 2;
    p.halo_tx1 = (g.tw + 2) * (g.th + 2) * p.kw1 * 2;
    p.a_slot_bytes = ((g.tw + 2) * (g.th + 2) * kw_max * 2 + 1023) / 1024 * 1024;
    stage_bytes = (block_n * kw_max * 2 + 1023) / 1024 * 1024;
    p.stage_bytes = stage_bytes;
    // Narrow N tiles (level 3: N = 64 / 80): the ncu source view shows BOTH single-thread roles saturated -- the producer
    // (one B tile of block_n box rows per tap) and the MMA issuer (~70 instructions per tap for 1-4 short MMAs) -- while
    // the tensor pipe idles.  Two CTAs per SM (the LIGHT instantiation: two producers, two issuers, staged epilogue)
    // double both; the shallower rings are what fits 2 x 104 KB.
    const int hl_budget = light_budget - 2 * p.a_slot_bytes;
    if (p.tmem_cols <= 256 && block_n <= 96 && hl_budget / stage_bytes >= 3) {
      light = true;
      p.a_slots = 2;
      p.b_off = p.a_slots * p.a_slot_bytes;
      stages = hl_budget / stage_bytes;
    } else {
      light = false;   // one CTA per SM with all of its shared memory
      p.a_slots = 3;
      p.b_off = p.a_slots * p.a_slot_bytes;
      stages = (TC_SMEM_BUDGET - p.b_off) / stage_bytes;
    }
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    if (stages < 3) return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): halo mode does not fit shared memory");
  }
  p.stages = stages;
  p.w_off = (g.halo ? p.b_off : 0) + stages * stage_bytes;
  p.epi_off = p.w_off + w_bytes;
  const bool staged = light && staged_out;
  const int64_t ktot = (int64_t)p.taps * (p.kpad0 + p.kpad1);

  int rc;
  const uint64_t esz = 2;
  if (g.cell) {
    // [c][dw=2][j=Wout][dh=2][ib=Hout*B]: output pixel (ib, j), tap (dh, dw) reads input pixel (2*ib + dh, 2*j + dw)
    // (rows of consecutive images are Hin input rows = Hout output rows apart, so (row, image) merge into one axis)
    const int rows = d.Hout * d.B;
    uint64_t dims[5] = {(uint64_t)d.c0, 2, (uint64_t)d.Wout, 2, (uint64_t)rows};
    uint64_t str[4] = {(uint64_t)d.ld0 * esz, 2ull * d.ld0 * esz, (uint64_t)d.Win * d.ld0 * esz,
                       2ull * d.Win * d.ld0 * esz};
    uint32_t box[5] = {(uint32_t)p.kw0, 1, (uint32_t)g.tw, 1, (uint32_t)g.th};
    if ((rc = encode_map(&p.tm_a0, d.a0, 5, dims, str, box, p.kw0)) != CCVPE_OK) return rc;
    p.a_rank = 5;
    p.tiles[0] = 1; p.tiles[1] = d.Wout / g.tw; p.tiles[2] = 1; p.tiles[3] = (rows + g.th - 1) / g.th;
    p.box[0] = 1; p.box[1] = g.tw; p.box[2] = 1; p.box[3] = g.th;
    for (int t = 0; t < 4; ++t) {
      p.tap_off[t][0] = t & 1;   // dw
      p.tap_off[t][1] = 0;
      p.tap_off[t][2] = t >> 1;  // dh
      p.tap_off[t][3] = 0;
    }
    p.out_stride[0] = 0; p.out_stride[1] = 1; p.out_stride[2] = 0; p.out_stride[3] = d.Wout;
    p.extent[0] = 1 << 30; p.extent[1] = d.Wout; p.extent[2] = 1 << 30; p.extent[3] = rows;
  } else if (d.kh == 1) {
    // 1x1 (transposed convs): the M axis is just the flattened pixel index -> 2-D maps, 128 consecutive pixels per tile
    const int64_t M = (int64_t)d.B * d.Hout * d.Wout;
    for (int s = 0; s < 2; ++s) {
      const void* base = s ? d.a1 : d.a0;
      const int c = s ? d.c1 : d.c0, ld = s ? d.ld1 : d.ld0;
      if (!c) continue;
      const int kw = s ? p.kw1 : p.kw0;
      uint64_t dims[2] = {(uint64_t)c, (uint64_t)M};
      uint64_t str[1] = {(uint64_t)ld * esz};
      uint32_t box[2] = {(uint32_t)kw, TC_BM};
      if ((rc = encode_map(s ? &p.tm_a1 : &p.tm_a0, base, 2, dims, str, box, kw)) != CCVPE_OK) return rc;
    }
    p.a_rank = 2;
    p.tiles[0] = (int)((M + TC_BM - 1) / TC_BM); p.tiles[1] = p.tiles[2] = p.tiles[3] = 1;
    p.box[0] = TC_BM; p.box[1] = p.box[2] = p.box[3] = 1;
    p.out_stride[0] = 1; p.out_stride[1] = p.out_stride[2] = p.out_stride[3] = 0;
    p.extent[0] = (int)M; p.extent[1] = p.extent[2] = p.extent[3] = 1;
  } else {
    p.a_rank = 4;
    for (int s = 0; s < 2; ++s) {
      const void* base = s ? d.a1 : d.a0;
      const int c = s ? d.c1 : d.c0, ld = s ? d.ld1 : d.ld0;
      if (!c) continue;
      uint64_t dims[4] = {(uint64_t)c, (uint64_t)d.Win, (uint64_t)d.Hin, (uint64_t)d.B};
      uint64_t str[3] = {(uint64_t)ld * esz, (uint64_t)d.Win * ld * esz, (uint64_t)d.Hin * d.Win * ld * esz};
      const int kw = s ? p.kw1 : p.kw0;
      uint32_t box[4] = {(uint32_t)kw, (uint32_t)(g.tw + (g.halo ? 2 : 0)), (uint32_t)(g.th + (g.halo ? 2 : 0)), (uint32_t)g.tb};
      if ((rc = encode_map(s ? &p.tm_a1 : &p.tm_a0, base, 4, dims, str, box, kw)) != CCVPE_OK) return rc;
    }
    p.tiles[0] = d.Wout / g.tw; p.tiles[1] = d.Hout / g.th; p.tiles[2] = (d.B + g.tb - 1) / g.tb; p.tiles[3] = 1;
    p.box[0] = g.tw; p.box[1] = g.th; p.box[2] = g.tb; p.box[3] = 1;
    for (int t = 0; t < p.taps; ++t) {
      p.tap_off[t][0] = (t % d.kw) - d.pad;
      p.tap_off[t][1] = (t / d.kw) - d.pad;
      p.tap_off[t][2] = 0;
      p.tap_off[t][3] = 0;
    }
    p.out_stride[0] = 1; p.out_stride[1] = d.Wout; p.out_stride[2] = d.Hout * d.Wout; p.out_stride[3] = 0;
    p.extent[0] = d.Wout; p.extent[1] = d.Hout; p.extent[2] = d.B; p.extent[3] = 1;
  }
  for (int s = 0; s < (d.c1 ? 2 : 1); ++s) {
    const int kw = s ? p.kw1 : p.kw0;
    uint64_t dims[2] = {(uint64_t)ktot, (uint64_t)d.N};
    uint64_t str[1] = {(uint64_t)ktot * esz};
    uint32_t box[2] = {(uint32_t)kw, (uint32_t)block_n};
    if ((rc = encode_map(s ? &p.tm_b1 : &p.tm_b0, d.w_nk, 2, dims, str, box, kw)) != CCVPE_OK) return rc;
  }
  const int m_tiles = p.tiles[0] * p.tiles[1] * p.tiles[2] * p.tiles[3];
  p.total_tiles = m_tiles * n_tiles_n;
  // the kernel decomposes tile / row indices with shifts: box[] are powers of two by construction, tiles[] too except the
  // last non-unit one, which takes whatever is left of the tile index
  {
    int last = 0;
    for (int i = 0; i < 4; ++i)
      if (p.tiles[i] > 1) last = i;
    for (int i = 0; i < 4; ++i) {
      if (!is_pow2(p.box[i]) || (i < last && !is_pow2(p.tiles[i])))
        return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): tile decomposition is not a power of two");
      p.box_shift[i] = ilog2(p.box[i]);
      p.tile_shift[i] = i < last ? ilog2(p.tiles[i]) : (i == last ? 30 : 0);
    }
  }
  fill_epi(p.e, d);
  if (out_pad) {
    if (d.relu != 2 || d.kh != 1)
      return fail(CCVPE_ERR_UNSUPPORTED, "ccvpe_igemm(tcgen05): padded output is a feature of the 1x1 SiLU epilogue");
    p.pad_w = d.Wout; p.pad_h = d.Hout; p.pad_wp = out_pad->Wp; p.pad_hp = out_pad->Hp; p.pad_lo = out_pad->lo;
  }

  const int smem = (g.halo ? p.b_off : 0) + stages * stage_bytes + w_bytes + (staged ? (TC_EPI_WARPS * EPI_WARP_STAGE_BYTES) : 0) + 1024;
  const int max_grid = (light ? 2 : 1) * sm_count();
  int grid = p.total_tiles < max_grid ? p.total_tiles : max_grid;
  if (p.w_resident) {   // whole groups of n_tiles_n CTAs, one per N tile
    int groups = max_grid / n_tiles_n;
    if (groups > m_tiles) groups = m_tiles;
    if (groups < 1) groups = 1;
    grid = groups * n_tiles_n;
  }
  cudaError_t attr_err = cudaSuccess;
#define CCVPE_LAUNCH_IGEMM(MODE, R1, F32)                                                                              \
  do {                                                                                                                 \
    static thread_local uint64_t attr_l = 0, attr_h = 0;                                                               \
    if (light) {                                                                                                       \
      if (first_use_on_device(attr_l)) {                                                                               \
        attr_err = cudaFuncSetAttribute(igemm_tcgen05_kernel<true, MODE, R1, F32>,                                     \
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);               \
      }                                                                                                                \
      igemm_tcgen05_kernel<true, MODE, R1, F32><<<grid, 64 + 32 * TC_EPI_WARPS, smem, st>>>(p);                         \
    } else {                                                                                                           \
      if (first_use_on_device(attr_h)) {                                                                               \
        attr_err = cudaFuncSetAttribute(igemm_tcgen05_kernel<false, MODE, R1, F32>,                                    \
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);               \
      }                                                                                                                \
      igemm_tcgen05_kernel<false, MODE, R1, F32><<<grid, 64 + 32 * TC_EPI_WARPS, smem, st>>>(p);                        \
    }                                                                                                                  \
  } while (0)
  if (epi_variant(p.e) == 6) {
    CCVPE_LAUNCH_IGEMM(3, false, false);
  } else {
    CCVPE_EPI_SWITCH(epi_variant(p.e), CCVPE_LAUNCH_IGEMM)
  }
#undef CCVPE_LAUNCH_IGEMM
  if (attr_err != cudaSuccess) return fail(CCVPE_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(attr_err));
  return check_launch("igemm_tcgen05_kernel");
}

}  // namespace ccvpe
