// a4/a5/a6 on tensor cores -- the rolled cosine correlation as a TMA-fed tcgen05 GEMM (bf16 path; full-circle L == C and
// windowed L < C: limited FoV, KITTI, Oxford's centred window).
//
//   dot[b, p, i] = sum_c x[b, p, c] * G[b, i, c],      G = banded circulant of the ground descriptor (match.cu)
//
// Pixels sit on the UMMA M axis (128 per tile), the R <= 32 orientations on N (padded to 32), channels on K.  A tiles
// [128 px x kw ch] arrive by 2-D TMA straight from the channels-last map, G tiles [32 x kw] likewise; accumulators live in
// TMEM (double buffered, 2 x 32 columns).  While the tensor pipe consumes a K block, four "norm" warps read the same
// shared-memory tile (one thread per pixel, chunk order rotated per row so the 128-bit loads are conflict free) and
// accumulate sum_c x^2, which gives both the cosine denominator and the 1/||x|| that F.normalize needs.  The same warps
// run the epilogue: tcgen05.ld -> divide -> planar fp32 score stores (one pixel per lane: coalesced per orientation),
// max over the selected orientations, 1/norm, and (bottleneck level only) the channels-last score copy and x-hat.
// Windowed levels (L < C) need one denominator PER ORIENTATION: sum of x^2 over the channels of window i.  Every window is
// a (circular) interval of channels, so its sum of squares is a difference of PREFIX sums: a norm thread walks its pixel's
// channels in order keeping the running sum, and drops a snapshot into shared memory at each of the <= 2R distinct window
// boundaries (positions are the same for every pixel: an 8-bit event mask per 16-byte chunk, tested on the uniform path;
// chunks without a boundary -- almost all of them -- take the plain 8-FMA path).  The epilogue forms
//     wsq[i] = P[end_i] - P[start_i]   (+ P[C] when the window wraps).
// Cost over the full-circle kernel: one table byte per chunk and <= 2R stores per pixel, whatever the window granularity.
// The correlation moves 2*R flops per loaded element (AI 8-20 flop/B in bf16) so the roofline that bounds it is HBM;
// the tensor pipe is what keeps the arithmetic off the critical path.
#include "tcgen05_common.cuh"

namespace ccvpe {

constexpr int MT_THREADS = 256;     // warps 0-3 control, 4-7 norm + epilogue
constexpr int MT_MAX_STAGES = 8;
constexpr int MT_N = 32;

struct MatchTcParams {
  CUtensorMap tm_x, tm_g;
  int kw, nb, C, HW, B, tiles_per_img, total_tiles, stages, a_bytes, stage_bytes;
  int n_rolls, ld_scores_cl;
  int L, offset, n_events;               // windowed: window length / first channel, distinct boundaries (host count)
  int shifts[32];                        // roll shifts (channels)
  uint32_t max_mask;
  const float* gnorm;
  const __nv_bfloat16* x;
  float* scores;
  __nv_bfloat16* scores_cl;
  float* max_out;
  float* inv_norm;
  __nv_bfloat16* xhat;
};

struct ShiftArg {
  int s[MT_N];
};

__global__ void build_rolled_descriptor_bf16_kernel(const float* __restrict__ g, int L, int C, int offset,
                                                    const ShiftArg shifts, int n_rolls,
                                                    __nv_bfloat16* __restrict__ G, float* __restrict__ gnorm) {
  const int b = blockIdx.y, i = blockIdx.x;
  if (i < MT_N) {
    __nv_bfloat16* row = G + ((int64_t)b * MT_N + i) * C;
    if (i < n_rolls) {
      const int base = ((offset + shifts.s[i]) % C + C) % C;
      for (int c = threadIdx.x; c < C; c += blockDim.x) {
        int k = c - base;
        if (k < 0) k += C;
        row[c] = __float2bfloat16_rn(k < L ? g[(int64_t)b * L + k] : 0.f);
      }
    } else {
      for (int c = threadIdx.x; c < C; c += blockDim.x) row[c] = __float2bfloat16_rn(0.f);
    }
  } else {
    __shared__ float red[32];
    float s = 0.f;
    for (int k = threadIdx.x; k < L; k += blockDim.x) {
      float v = g[(int64_t)b * L + k];
      s = fmaf(v, v, s);
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
      float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
      t = warp_sum(t);
      if (threadIdx.x == 0) gnorm[b] = sqrtf(t);
    }
  }
}

constexpr int MT_WMAX = 24;              // orientations of a windowed level (C ABI limit)
constexpr int MT_MAX_EVENTS = 2 * MT_WMAX;
constexpr int MT_MAX_CHUNKS = 2048 / 8 + 8;   // 16-byte chunks of a pixel (C <= 2048, padded to the K-block width)

template <bool WINDOWED>
__global__ void __launch_bounds__(MT_THREADS, WINDOWED ? 3 : 4) match_tcgen05_kernel(const __grid_constant__ MatchTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[MT_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_empty[MT_MAX_STAGES];
  __shared__ __align__(8) uint64_t bar_tmem_full[2];
  __shared__ __align__(8) uint64_t bar_tmem_empty[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_empty[s]), 1 + 4);     // MMA commit + one arrival per norm warp
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tmem_full[a]), 1);
      mbar_init(smem_u32(&bar_tmem_empty[a]), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tm_x);
    prefetch_tmap(&p.tm_g);
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"(64)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // ---- windowed: boundary events (identical for every pixel of the level) ----
  __shared__ uint32_t s_posbits[2048 / 32 + 1];      // bit p set: a window starts or ends at channel position p (0 < p < C)
  __shared__ uint16_t s_wordrank[2048 / 32 + 1];     // number of events below word w
  __shared__ uint8_t s_evmask[MT_MAX_CHUNKS];        // per chunk: bit t set = snapshot after element t of the chunk
  __shared__ uint8_t s_evbase[MT_MAX_CHUNKS];        // index of the chunk's first snapshot
  __shared__ int8_t s_roll_a[MT_WMAX], s_roll_b[MT_WMAX], s_roll_wrap[MT_WMAX];   // snapshot ids: -1 = P[0] = 0, -2 = P[C]
  float* s_snap = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)) + p.stages * p.stage_bytes);
  if (WINDOWED) {
    const int n_words = (p.C + 31) >> 5;
    for (int w = threadIdx.x; w <= n_words; w += MT_THREADS) s_posbits[w] = 0u;
    __syncthreads();
    if ((int)threadIdx.x < p.n_rolls) {
      const int base = ((p.offset + p.shifts[threadIdx.x]) % p.C + p.C) % p.C;
      int end = base + p.L;
      if (end >= p.C) end -= p.C;                    // end == C maps to position 0 of the wrapped copy: handled as P[C]
      if (base) atomicOr(&s_posbits[base >> 5], 1u << (base & 31));
      if (end) atomicOr(&s_posbits[end >> 5], 1u << (end & 31));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int acc = 0;
      for (int w = 0; w <= n_words; ++w) {
        s_wordrank[w] = (uint16_t)acc;
        acc += __popc(s_posbits[w]);
      }
    }
    __syncthreads();
    auto rank_of = [&](int pos) { return (int)s_wordrank[pos >> 5] + __popc(s_posbits[pos >> 5] & ((1u << (pos & 31)) - 1u)); };
    if ((int)threadIdx.x < p.n_rolls) {
      const int base = ((p.offset + p.shifts[threadIdx.x]) % p.C + p.C) % p.C;
      const int end = base + p.L;
      s_roll_a[threadIdx.x] = (int8_t)(base ? rank_of(base) : -1);
      s_roll_wrap[threadIdx.x] = (int8_t)(end > p.C ? 1 : 0);
      s_roll_b[threadIdx.x] = (int8_t)(end == p.C ? -2 : rank_of(end > p.C ? end - p.C : end));
    }
    const int n_chunks = (p.nb * p.kw) >> 3;
    for (int ch = threadIdx.x; ch < n_chunks; ch += MT_THREADS) {
      // snapshot after element t of chunk ch <=> boundary at position ch*8 + t + 1
      const int p0 = ch * 8 + 1;
      uint32_t bits = 0;
      if (p0 < p.C + 8) {
        const int w = p0 >> 5, sft = p0 & 31;
        uint64_t two = (uint64_t)s_posbits[w < n_words + 1 ? w : n_words];
        if (w + 1 <= n_words) two |= (uint64_t)s_posbits[w + 1] << 32;
        bits = (uint32_t)(two >> sft) & 0xffu;
      }
      s_evmask[ch] = (uint8_t)bits;
      s_evbase[ch] = (uint8_t)(p0 < p.C ? rank_of(p0) : 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged, single-lane issue via elect_one) =====================
    {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx = (uint32_t)((TC_BM + MT_N) * p.kw * 2);
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int b = tile / p.tiles_per_img;
        const int prow = b * p.HW + (tile - b * p.tiles_per_img) * TC_BM;   // first pixel row of the tile
        for (int kb = 0; kb < p.nb; ++kb) {
          mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
          if (elect_one()) {
            const uint32_t full = smem_u32(&bar_full[stage]);
            const uint32_t dst = smem_base + (uint32_t)(stage * p.stage_bytes);
            mbar_arrive_expect_tx(full, tx);
            tma_load_2d(dst, &p.tm_x, full, kb * p.kw, prow);
            tma_load_2d(dst + (uint32_t)p.a_bytes, &p.tm_g, full, kb * p.kw, b * MT_N);
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (converged warp, elect_one issue) =====================
    {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(MT_N >> 3) << 17) |
                             ((uint32_t)(TC_BM >> 4) << 24);
      const uint64_t hi = (uint64_t)(uint32_t)(make_smem_desc(0, p.kw) >> 32) << 32;
      const int nfull = p.kw >> 4, ntail = (p.C - (p.nb - 1) * p.kw + 15) >> 4;
      const uint32_t lo_base = ((smem_base & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t lo_stage = (uint32_t)p.stage_bytes >> 4, lo_b = (uint32_t)p.a_bytes >> 4;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = (uint32_t)it & 1u;
        mbar_wait(smem_u32(&bar_tmem_empty[acc]), (((uint32_t)it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * (uint32_t)MT_N;
        uint32_t accumulate = 0;
#pragma unroll 1
        for (int kb = 0; kb < p.nb; ++kb) {
          const int nk16 = (kb == p.nb - 1) ? ntail : nfull;
          mbar_wait(smem_u32(&bar_full[stage]), phase);
          tc_fence_after();
          const uint32_t a_lo = lo_base + (uint32_t)stage * lo_stage;
          const uint64_t adesc = hi | a_lo, bdesc = hi | (a_lo + lo_b);
          if (elect_one()) {
            umma_bf16(tmem_d, adesc, bdesc, idesc, accumulate);
            if (nk16 > 1) umma_bf16(tmem_d, adesc + 2, bdesc + 2, idesc, 1u);
            if (nk16 > 2) umma_bf16(tmem_d, adesc + 4, bdesc + 4, idesc, 1u);
            if (nk16 > 3) umma_bf16(tmem_d, adesc + 6, bdesc + 6, idesc, 1u);
            umma_commit(smem_u32(&bar_empty[stage]));
          }
          accumulate = 1;
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (elect_one()) umma_commit(smem_u32(&bar_tmem_full[acc]));
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===================== norm + epilogue warps: thread = pixel row of the tile =====================
    const int ew = warp & 3;
    const int row = ew * 32 + lane;
    const int row_bytes = p.kw * 2;
    const int chunks = row_bytes >> 4;                    // 16-byte chunks per row: 2, 4 or 8
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const int b = tile / p.tiles_per_img;
      const int pix = (tile - b * p.tiles_per_img) * TC_BM + row;     // pixel within the image
      const bool valid = pix < p.HW;
      float sq = 0.f;
      // inverse of the TMA swizzle: 16-byte chunk position within the row ^ swz = logical chunk (128B / 64B / 32B swizzle)
      const int swz = p.kw == 64 ? (row & 7) : (p.kw == 32 ? ((row >> 1) & 3) : ((row >> 2) & 1));
      float* snap = s_snap + row;                      // snapshot e of this pixel: snap[e * 128]
#pragma unroll 1
      for (int kb = 0; kb < p.nb; ++kb) {
        mbar_wait(smem_u32(&bar_full[stage]), phase);
        const uint8_t* tile_ptr = smem_raw + (smem_base - smem_u32(smem_raw)) + stage * p.stage_bytes + row * row_bytes;
        float s0 = WINDOWED ? sq : 0.f, s1 = 0.f;
        for (int j = 0; j < chunks; ++j) {
          // full circle: rotate the chunk order by the row index: lanes of a warp then cover all bank groups (conflict
          // free); the swizzle only permutes chunks inside a row, and a sum of squares does not care about their order.
          // Windowed: every lane reads LOGICAL chunk j (physical j ^ swz -- conflict free by construction of the
          // swizzle): channels are visited in order, so the running sum is the prefix sum the window boundaries need.
          const int phys = WINDOWED ? (j ^ swz) : ((j + row) & (chunks - 1));
          const uint4 q = *reinterpret_cast<const uint4*>(tile_ptr + (phys << 4));
          const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.x));
          const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.y));
          const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.z));
          const float2 f3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.w));
          if (WINDOWED) {
            const int gch = kb * chunks + j;
            const uint32_t ev = s_evmask[gch];         // warp-uniform
            if (ev == 0u) {
              s0 = fmaf(f0.x, f0.x, s0); s0 = fmaf(f0.y, f0.y, s0);
              s0 = fmaf(f1.x, f1.x, s0); s0 = fmaf(f1.y, f1.y, s0);
              s0 = fmaf(f2.x, f2.x, s0); s0 = fmaf(f2.y, f2.y, s0);
              s0 = fmaf(f3.x, f3.x, s0); s0 = fmaf(f3.y, f3.y, s0);
            } else {
              int e = s_evbase[gch];
              const float el[8] = {f0.x, f0.y, f1.x, f1.y, f2.x, f2.y, f3.x, f3.y};
#pragma unroll
              for (int t = 0; t < 8; ++t) {
                s0 = fmaf(el[t], el[t], s0);
                if ((ev >> t) & 1u) {                  // uniform
                  snap[e * TC_BM] = s0;
                  ++e;
                }
              }
            }
          } else {
            s0 = fmaf(f0.x, f0.x, s0); s1 = fmaf(f0.y, f0.y, s1);
            s0 = fmaf(f1.x, f1.x, s0); s1 = fmaf(f1.y, f1.y, s1);
            s0 = fmaf(f2.x, f2.x, s0); s1 = fmaf(f2.y, f2.y, s1);
            s0 = fmaf(f3.x, f3.x, s0); s1 = fmaf(f3.y, f3.y, s1);
          }
        }
        if (WINDOWED) sq = s0;                         // (running prefix: carried across K blocks)
        else sq += s0 + s1;
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bar_empty[stage]));
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      // ---- epilogue ----
      const uint32_t acc = (uint32_t)it & 1u;
      mbar_wait(smem_u32(&bar_tmem_full[acc]), ((uint32_t)it >> 1) & 1u);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + acc * (uint32_t)MT_N, v);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bar_tmem_empty[acc]));   // accumulator is in registers: release it early
      if (valid) {
        const float nrm = sqrtf(sq);
        const float inv = 1.f / fmaxf(nrm, 1e-12f);
        // one reciprocal of the cosine denominator, no epsilon: den == 0 gives inf and 0 * inf = NaN like the
        // reference's 0 / 0 (models.py:196)
        const float gn = __ldg(p.gnorm + b);
        const float rden = 1.f / (nrm * gn);
        const float rgn = 1.f / gn;
        const int64_t gp = (int64_t)b * p.HW + pix;
        float best = -INFINITY;
        bool any_nan = false;
        float sc[MT_N];
        float* sp = p.scores ? p.scores + (int64_t)b * p.n_rolls * p.HW + pix : nullptr;
#pragma unroll
        for (int i = 0; i < MT_N; ++i) {
          if (i < p.n_rolls) {
            if (WINDOWED && i < MT_WMAX) {
              // windowed cosine denominator sqrt(sum_window x^2) * ||g|| from the prefix-sum snapshots; a zero window gives
              // 0 * inf = NaN like the reference's 0 / 0 (models.py:196)
              const int ia = s_roll_a[i], ib = s_roll_b[i];
              const float pa = ia < 0 ? 0.f : snap[ia * TC_BM];
              const float pb = ib == -2 ? sq : (ib < 0 ? 0.f : snap[ib * TC_BM]);
              const float wsq = s_roll_wrap[i] ? (sq - pa) + pb : pb - pa;
              sc[i] = __uint_as_float(v[i]) * (rsqrtf(fmaxf(wsq, 0.f)) * rgn);
            } else {
              sc[i] = __uint_as_float(v[i]) * rden;
            }
            if (sp) sp[(int64_t)i * p.HW] = sc[i];
            if ((p.max_mask >> i) & 1u) {
              any_nan |= (sc[i] != sc[i]);
              best = fmaxf(best, sc[i]);
            }
          } else {
            sc[i] = 0.f;
          }
        }
        if (any_nan) best = __int_as_float(0x7fc00000);
        if (p.max_out) p.max_out[gp] = best;
        if (p.inv_norm) p.inv_norm[gp] = inv;
        if (p.scores_cl) {
          __nv_bfloat16* dst = p.scores_cl + gp * p.ld_scores_cl;
#pragma unroll
          for (int i = 0; i < MT_N; i += 8) {
            if (i < p.ld_scores_cl) {
              uint4 pk;
              __nv_bfloat162 q0 = __floats2bfloat162_rn(sc[i + 0], sc[i + 1]), q1 = __floats2bfloat162_rn(sc[i + 2], sc[i + 3]);
              __nv_bfloat162 q2 = __floats2bfloat162_rn(sc[i + 4], sc[i + 5]), q3 = __floats2bfloat162_rn(sc[i + 6], sc[i + 7]);
              pk.x = *reinterpret_cast<uint32_t*>(&q0);
              pk.y = *reinterpret_cast<uint32_t*>(&q1);
              pk.z = *reinterpret_cast<uint32_t*>(&q2);
              pk.w = *reinterpret_cast<uint32_t*>(&q3);
              *reinterpret_cast<uint4*>(dst + i) = pk;
            }
          }
          for (int i = MT_N; i < p.ld_scores_cl; ++i) dst[i] = __float2bfloat16_rn(0.f);
        }
        if (p.xhat) {   // bottleneck level only (64 pixels per image): one more read of this pixel's vector
          const __nv_bfloat16* src = p.x + gp * p.C;
          __nv_bfloat16* dst = p.xhat + gp * p.C;
          for (int c = 0; c < p.C; c += 8) {
            uint4 q = *reinterpret_cast<const uint4*>(src + c);
            __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float2 f = __bfloat1622float2(h[j]);
              h[j] = __floats2bfloat162_rn(f.x * inv, f.y * inv);
            }
            *reinterpret_cast<uint4*>(dst + c) = q;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(64) : "memory");
  }
}

static int count_window_events(int C, int L, int offset, const int32_t* shifts_host, int n_rolls) {
  if (L == C) return 0;
  int pos[2 * MT_WMAX], n = 0;
  for (int i = 0; i < n_rolls && i < MT_WMAX; ++i) {
    const int base = ((offset + shifts_host[i]) % C + C) % C;
    int end = base + L;
    if (end >= C) end -= C;
    const int cand[2] = {base, end};
    for (int k = 0; k < 2; ++k) {
      if (cand[k] == 0) continue;
      bool seen = false;
      for (int j = 0; j < n; ++j) seen |= (pos[j] == cand[k]);
      if (!seen) pos[n++] = cand[k];
    }
  }
  return n;
}

bool match_tcgen05_supported(int dtype, int C, int L, int offset, const int32_t* shifts_host, int n_rolls,
                             int ld_scores_cl) {
  if (!(dtype == CCVPE_BF16 && L <= C && C % 8 == 0 && n_rolls <= MT_N && ld_scores_cl % 8 == 0)) return false;
  if (L == C) return true;
  return n_rolls <= MT_WMAX && C <= 2048;
}

// scratch layout (bytes from `scratch`): G bf16 [B, 32, C] | gnorm fp32 [B]
int match_tcgen05(const void* x, int B, int HW, int C, const float* g, int L, int offset, const int32_t* shifts_host,
                  int n_rolls, uint32_t max_mask, float* scores, void* scores_cl, int ld_scores_cl, float* max_out,
                  float* inv_norm, void* xhat, float* scratch, cudaStream_t st) {
  auto up = [](int64_t v) { return (v + 255) / 256 * 256; };
  uint8_t* base = reinterpret_cast<uint8_t*>(scratch);
  __nv_bfloat16* G = reinterpret_cast<__nv_bfloat16*>(base);
  float* gnorm = reinterpret_cast<float*>(base + up((int64_t)B * MT_N * C * 2));
  const bool windowed = L < C;
  const int n_events = count_window_events(C, L, offset, shifts_host, n_rolls);
  ShiftArg sa;   // the roll table travels as a kernel argument (no copy, no sync, graph-capturable)
  for (int i = 0; i < MT_N; ++i) sa.s[i] = i < n_rolls ? shifts_host[i] : 0;
  build_rolled_descriptor_bf16_kernel<<<dim3(MT_N + 1, B), 256, 0, st>>>(g, L, C, offset, sa, n_rolls, G, gnorm);
  int rc = check_launch("build_rolled_descriptor_bf16_kernel");
  if (rc != CCVPE_OK) return rc;

  static thread_local MatchTcParams p;
  memset(&p, 0, sizeof(p));
  p.kw = tc_block_width(C);
  p.nb = (C + p.kw - 1) / p.kw;
  p.C = C;
  p.HW = HW;
  p.B = B;
  p.tiles_per_img = (HW + TC_BM - 1) / TC_BM;
  p.total_tiles = B * p.tiles_per_img;
  p.a_bytes = TC_BM * p.kw * 2;
  p.stage_bytes = p.a_bytes + ((MT_N * p.kw * 2 + 1023) / 1024) * 1024;
  // ~52 KB of pipeline per CTA so that four CTAs (16 norm/epilogue warps) share an SM: the epilogue is scalar-ALU and
  // store bound and needs the extra warps to hide its own latency (windowed: three CTAs per SM, each with up to 24 KB of
  // prefix-sum snapshots behind its ring)
  // The coarse levels have fewer tiles than the GPU has CTA slots (level 1 of a batch of 64: 64 tiles of 20 K blocks): there
  // a CTA is alone on its SM and a two-stage ring exposes the full load latency on every K block (52 us for 42 MB) -- give
  // it the ring depth the empty SM can afford instead.
  const int per_sm_max = windowed ? 3 : 4;
  int ctas_needed = (p.total_tiles + sm_count() - 1) / sm_count();
  if (ctas_needed > per_sm_max) ctas_needed = per_sm_max;
  const int snap_bytes = windowed ? (n_events > 0 ? n_events : 1) * TC_BM * 4 : 0;
  const int budget = ctas_needed >= per_sm_max ? 52 * 1024 : (160 * 1024) / ctas_needed - snap_bytes;
  int stages = budget / p.stage_bytes;
  if (stages < 2) stages = 2;
  p.stages = stages > MT_MAX_STAGES ? MT_MAX_STAGES : stages;
  p.n_rolls = n_rolls;
  p.ld_scores_cl = scores_cl ? ld_scores_cl : 0;
  p.L = L;
  p.offset = offset;
  p.n_events = n_events;
  for (int i = 0; i < 32; ++i) p.shifts[i] = sa.s[i];
  p.max_mask = max_mask;
  p.gnorm = gnorm;
  p.x = static_cast<const __nv_bfloat16*>(x);
  p.scores = scores;
  p.scores_cl = static_cast<__nv_bfloat16*>(scores_cl);
  p.max_out = max_out;
  p.inv_norm = inv_norm;
  p.xhat = static_cast<__nv_bfloat16*>(xhat);
  {
    uint64_t dims[2] = {(uint64_t)C, (uint64_t)B * HW};
    uint64_t str[1] = {(uint64_t)C * 2};
    uint32_t box[2] = {(uint32_t)p.kw, TC_BM};
    if ((rc = encode_map(&p.tm_x, x, 2, dims, str, box, p.kw)) != CCVPE_OK) return rc;
    uint64_t gdims[2] = {(uint64_t)C, (uint64_t)B * MT_N};
    uint32_t gbox[2] = {(uint32_t)p.kw, MT_N};
    if ((rc = encode_map(&p.tm_g, G, 2, gdims, str, gbox, p.kw)) != CCVPE_OK) return rc;
  }
  const int smem = p.stages * p.stage_bytes + 1024 + (windowed ? (n_events > 0 ? n_events : 1) * TC_BM * 4 : 0);
  static thread_local uint64_t attr_set = 0;
  if (first_use_on_device(attr_set)) {
    cudaError_t e = cudaFuncSetAttribute(match_tcgen05_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 170 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(match_tcgen05_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 170 * 1024);
    if (e != cudaSuccess) return fail(CCVPE_ERR_CUDA, "cudaFuncSetAttribute(match): %s", cudaGetErrorString(e));
  }
  const int per_sm = windowed ? 3 : 4;
  const int grid = p.total_tiles < per_sm * sm_count() ? p.total_tiles : per_sm * sm_count();
  if (windowed) match_tcgen05_kernel<true><<<grid, MT_THREADS, smem, st>>>(p);
  else match_tcgen05_kernel<false><<<grid, MT_THREADS, smem, st>>>(p);
  return check_launch("match_tcgen05_kernel");
}

}  // namespace ccvpe
