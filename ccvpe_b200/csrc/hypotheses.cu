// Pose hypotheses: the k strongest mutually exclusive location modes of each heatmap, with the probability mass each one
// claims and the orientation at its pixel (semantics in include/ccvpe_b200.h, ccvpe_pose_hypotheses).
//
// One 8-CTA thread-block cluster per pair.  CTA c owns the band of rows [c*R, (c+1)*R), R = ceil(H/8), and holds it in
// shared memory with one halo row above and below (128 KiB + 4 KiB for a 512x512 map), loaded once with bulk copies, so the
// heatmap is read from HBM once.  Two bitmasks per band row: `claimed` (every pixel some disc covered) and `avail` (modes
// not yet claimed).  Each warp keeps the best key of the available modes in its rows in a register; a claim only removes
// candidates, so a warp rescans only when its own best was claimed.  A round:
//   1. every warp reads the 8 CTA bests of the previous round through distributed shared memory and takes their maximum,
//      the round's hypothesis (the same in every CTA, so every CTA stops in the same round);
//   2. every CTA claims its part of the disc and sums the newly claimed values in float64;
//   3. stale warps rescan, the CTA writes its new best (double-buffered by round parity, so one barrier per round
//      suffices) and its mass partial (one slot per round), and the cluster barrier publishes both.
// After the last round CTA 0 writes every hypothesis in parallel, one thread per slot: it folds the 8 mass partials in
// CTA order and reads `ori` at the hypothesis's pixel only; nothing of that sits in the rounds' critical path.
// The work of a round is split over the threads as a function of (pixel, radius, band) only and every sum is a fixed
// tree, so the output is a function of the map alone.  No workspace, no allocation, no host synchronisation.
#include "tcgen05_common.cuh"

namespace ccvpe {
namespace {

constexpr int kHypCtas = 8;               // CTAs per cluster = bands per map
constexpr int kHypWarps = 32;
constexpr int kHypThreads = 32 * kHypWarps;
constexpr int kHypMaxK = 64;
constexpr int kHypMaxRadius = 32767;
// opt-in shared memory of one block on sm_100 (227 KiB) less 2 KiB for the kernel's static shared memory
constexpr int64_t kHypSmemMax = 232448 - 2048;
constexpr uint32_t kHypChunk = 32768;     // bytes per bulk copy
constexpr uint64_t kPoison = ~0ull;       // a CTA best that means "this band holds a NaN"

struct HypGeom {
  int R, words;                           // rows per band, 32-bit mask words per row
  int64_t vals_bytes, bytes;              // band values (with halos and the 16-byte phase offset), total dynamic smem
};

__host__ __device__ inline HypGeom hyp_geom(int H, int W) {
  HypGeom g;
  g.R = (H + kHypCtas - 1) / kHypCtas;
  g.words = (W + 31) / 32;
  g.vals_bytes = (((int64_t)(g.R + 2) * W + 3) * 4 + 15) / 16 * 16;
  g.bytes = g.vals_bytes + 2 * 4 * (int64_t)g.R * g.words;
  return g;
}

// Candidates order by value, highest first, then by the smaller flat index: the larger key wins.  -0 and +0 get one key
// (they compare equal in NumPy's order); no candidate is key 0, which no value reaches (-inf gives 0x007fffff'...).
__device__ __forceinline__ uint64_t hyp_key(float v, int idx) {
  uint32_t u = __float_as_uint(v == 0.f ? 0.f : v);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((uint64_t)u << 32) | (uint32_t)~(uint32_t)idx;
}
__device__ __forceinline__ int key_idx(uint64_t key) { return (int)~(uint32_t)key; }

__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const uint64_t w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// every thread of every CTA of the cluster: shared-memory writes before it are visible to remote reads after it
__device__ __forceinline__ void cluster_sync() {
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint64_t ld_cluster_u64(const void* p, uint32_t rank) {
  uint32_t a;
  uint64_t v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
  asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

struct Band {
  const float* v;                         // v[(i - lo) * W + j] = h[i, j] for loaded rows lo <= i < hi
  uint32_t* claimed;
  uint32_t* avail;
  int r0, r1, lo, W, words;
  __device__ __forceinline__ float at(int i, int j) const { return v[(i - lo) * W + j]; }
};

// best key of the available modes in this warp's rows (band rows warp, warp + 32, ...), in every lane
__device__ uint64_t warp_best(const Band& s, int warp, int lane) {
  uint64_t best = 0;
  for (int ii = warp; ii < s.r1 - s.r0; ii += kHypWarps) {
    const int i = s.r0 + ii;
    for (int q = lane; q < s.words; q += 32) {
      uint32_t m = s.avail[ii * s.words + q];
      while (m) {
        const int j = q * 32 + __ffs(m) - 1;
        m &= m - 1;
        const uint64_t key = hyp_key(s.at(i, j), i * s.W + j);
        best = key > best ? key : best;
      }
    }
  }
  return warp_max_u64(best);
}

__global__ void __cluster_dims__(kHypCtas, 1, 1) __launch_bounds__(kHypThreads, 1)
pose_hypotheses_kernel(const float* __restrict__ heat, const float* __restrict__ ori, int H, int W, int k, int radius,
                       int64_t* __restrict__ idx_out, int32_t* __restrict__ rc_out, float* __restrict__ value_out,
                       float* __restrict__ mass_out, float* __restrict__ cs_out, double* __restrict__ angle_out,
                       uint8_t* __restrict__ valid_out, int32_t* __restrict__ count_out) {
  extern __shared__ __align__(16) uint8_t hyp_smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint64_t warp_key[kHypWarps];
  __shared__ double warp_mass[kHypWarps];
  __shared__ uint64_t cta_best[2];        // by round parity
  __shared__ uint64_t cta_mass[kHypMaxK]; // float64 bits of this band's mass partial, by round
  __shared__ int hyp_idx[kHypMaxK];       // the flat index of each round's hypothesis

  const uint32_t rank = cluster_rank();
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const HypGeom g = hyp_geom(H, W);
  const int64_t n = (int64_t)H * W;
  const float* hb = heat + (int64_t)b * n;

  Band s;
  s.r0 = min((int)rank * g.R, H);
  s.r1 = min(s.r0 + g.R, H);
  s.lo = max(s.r0 - 1, 0);
  s.W = W;
  s.words = g.words;
  s.claimed = reinterpret_cast<uint32_t*>(hyp_smem + g.vals_bytes);
  s.avail = s.claimed + g.R * g.words;

  // ---- load the band and its halo rows: bulk copies of the 16-byte aligned middle, plain loads of the <= 3 + 3 ends ----
  {
    const int hi = min(s.r1 + 1, H);
    const float* src = hb + (int64_t)s.lo * W;
    const int cnt = s.r1 > s.r0 ? (hi - s.lo) * W : 0;
    const int phase = (int)((reinterpret_cast<uintptr_t>(src) >> 2) & 3);
    float* dst = reinterpret_cast<float*>(hyp_smem) + phase;           // dst[e] has the 16-byte phase of src[e]
    s.v = dst;
    const int ea = min((4 - phase) & 3, cnt), eb = ea + (cnt - ea) / 4 * 4;
    const uint32_t bytes = (uint32_t)(eb - ea) * 4u;
    const uint32_t mbar = smem_u32(&bar);
    if (threadIdx.x == 0 && bytes) {
      mbar_init(mbar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      mbar_arrive_expect_tx(mbar, bytes);
      for (uint32_t off = 0; off < bytes; off += kHypChunk)
        bulk_load(smem_u32(dst + ea) + off, src + ea + off / 4, min(kHypChunk, bytes - off), mbar);
    }
    const int tid = (int)threadIdx.x;
    if (tid < ea) dst[tid] = src[tid];
    if (eb + tid < cnt) dst[eb + tid] = src[eb + tid];
    __syncthreads();                                                     // the barrier's init precedes every wait
    if (bytes) mbar_wait(mbar, 0);
    __syncthreads();
  }

  // ---- modes (>= every in-bounds 8-neighbour) and the NaN test, one warp per 32-pixel word ----
  bool has_nan = false;
  for (int u = warp; u < (s.r1 - s.r0) * g.words; u += kHypWarps) {
    const int ii = u / g.words, q = u - ii * g.words, i = s.r0 + ii, j = q * 32 + lane;
    bool mode = false, nan = false;
    if (j < W) {
      const float v = s.at(i, j);
      nan = v != v;
      mode = true;
#pragma unroll
      for (int di = -1; di <= 1; ++di)
#pragma unroll
        for (int dj = -1; dj <= 1; ++dj)
          if ((di || dj) && i + di >= 0 && i + di < H && j + dj >= 0 && j + dj < W) mode &= v >= s.at(i + di, j + dj);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, mode);
    has_nan |= __any_sync(0xffffffffu, nan);
    if (lane == 0) {
      s.avail[u] = m;
      s.claimed[u] = 0u;
    }
  }
  __syncthreads();
  uint64_t wk = has_nan ? kPoison : warp_best(s, warp, lane);           // this warp's best, kept across rounds
  if (lane == 0) warp_key[warp] = wk;
  __syncthreads();
  if (warp == 0) {
    const uint64_t c = warp_max_u64(warp_key[lane]);
    if (lane == 0) cta_best[0] = c;
  }
  cluster_sync();

  const int64_t r2 = (int64_t)radius * radius;
  const int64_t slot0 = (int64_t)b * k;
  int t = 0;
  for (; t < k; ++t) {
    const uint64_t best = warp_max_u64(lane < kHypCtas ? ld_cluster_u64(&cta_best[t & 1], lane) : 0ull);
    if (best == 0ull || best == kPoison) break;                        // no candidate left, or a NaN map (round 0 only)
    const int p = key_idx(best), i0 = p / W, j0 = p - i0 * W;
    if (threadIdx.x == 0) hyp_idx[t] = p;

    // claim the disc's part in this band; sum what no earlier hypothesis claimed
    double acc = 0.0;
    const int ca = max(i0 - radius, s.r0), cb = min(i0 + radius, s.r1 - 1);
    const int qa = max(j0 - radius, 0) >> 5, nq = (min(j0 + radius, W - 1) >> 5) - qa + 1;
    for (int u = warp; u < (cb - ca + 1) * nq; u += kHypWarps) {       // no iteration when ca > cb
      const int i = ca + u / nq, q = qa + u % nq, j = q * 32 + lane;
      const int w = (i - s.r0) * g.words + q;
      const int64_t di = i - i0, dj = j - j0;
      const uint32_t old = s.claimed[w];
      const uint32_t disc = __ballot_sync(0xffffffffu, j < W && di * di + dj * dj <= r2);
      if (((disc & ~old) >> lane) & 1u) acc += (double)s.at(i, j);
      __syncwarp();
      if (lane == 0) {
        s.claimed[w] = old | disc;
        s.avail[w] &= ~disc;
      }
    }
    acc = warp_sum_f64(acc);
    if (lane == 0) warp_mass[warp] = acc;
    __syncthreads();

    if (wk != 0ull) {                                                  // rescan only if this warp's best was claimed
      const int pw = key_idx(wk), iw = pw / W, jw = pw - iw * W;
      if (!((s.avail[(iw - s.r0) * g.words + (jw >> 5)] >> (jw & 31)) & 1u)) wk = warp_best(s, warp, lane);
    }
    if (lane == 0) warp_key[warp] = wk;
    __syncthreads();
    if (warp == 0) {
      const uint64_t c = warp_max_u64(warp_key[lane]);
      const double m = warp_sum_f64(warp_mass[lane]);
      if (lane == 0) {
        cta_best[(t + 1) & 1] = c;
        cta_mass[t] = (uint64_t)__double_as_longlong(m);
      }
    }
    cluster_sync();
  }

  // ---- CTA 0 writes the hypotheses, one thread per slot: fold the 8 mass partials in CTA order, read ori at the pixel ----
  if (rank == 0) {
    const float fnan = __int_as_float(0x7fc00000);
    for (int e = (int)threadIdx.x; e < t; e += kHypThreads) {
      double mass = 0.0;
      for (uint32_t c = 0; c < kHypCtas; ++c) mass += __longlong_as_double((long long)ld_cluster_u64(&cta_mass[e], c));
      const int p = hyp_idx[e], i0 = p / W;
      const int64_t o = slot0 + e;
      idx_out[o] = p;
      rc_out[2 * o + 0] = i0;
      rc_out[2 * o + 1] = p - i0 * W;
      value_out[o] = hb[p];
      mass_out[o] = __double2float_rn(mass);
      const float c = ori[((int64_t)b * 2 + 0) * n + p], sn = ori[((int64_t)b * 2 + 1) * n + p];
      cs_out[2 * o + 0] = c;
      cs_out[2 * o + 1] = sn;
      bool ok;
      angle_out[o] = pose_angle_deg(c, sn, ok);
      valid_out[o] = ok ? 1 : 0;
    }
    for (int e = t + (int)threadIdx.x; e < k; e += kHypThreads) {
      const int64_t o = slot0 + e;
      idx_out[o] = -1;
      rc_out[2 * o + 0] = -1;
      rc_out[2 * o + 1] = -1;
      value_out[o] = fnan;
      mass_out[o] = fnan;
      cs_out[2 * o + 0] = fnan;
      cs_out[2 * o + 1] = fnan;
      angle_out[o] = __longlong_as_double(0x7ff8000000000000LL);
      valid_out[o] = 0;
    }
    if (threadIdx.x == 0) count_out[b] = t;
  }
  cluster_sync();                                                      // no CTA exits while CTA 0 may still read it
}

}  // namespace
}  // namespace ccvpe

extern "C" int64_t ccvpe_pose_hypotheses_smem_bytes(int H, int W) {
  if (H <= 0 || W <= 0) return -1;
  const ccvpe::HypGeom g = ccvpe::hyp_geom(H, W);
  return g.bytes <= ccvpe::kHypSmemMax ? g.bytes : -1;
}

extern "C" int ccvpe_pose_hypotheses(const float* heatmap, const float* ori, int B, int H, int W, int k, int radius,
                                     int64_t* idx, int32_t* rc, float* value, float* mass, float* cs, double* angle_deg,
                                     uint8_t* valid, int32_t* count, void* stream) {
  using namespace ccvpe;
  CCVPE_REQUIRE(heatmap && ori && idx && rc && value && mass && cs && angle_deg && valid && count,
                "ccvpe_pose_hypotheses: null pointer");
  CCVPE_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0, "ccvpe_pose_hypotheses: bad shape B=%d H=%d W=%d", B, H, W);
  CCVPE_REQUIRE(k >= 1 && k <= kHypMaxK, "ccvpe_pose_hypotheses: k=%d outside [1, %d]", k, kHypMaxK);
  CCVPE_REQUIRE(radius >= 0 && radius <= kHypMaxRadius, "ccvpe_pose_hypotheses: radius=%d outside [0, %d]", radius,
                kHypMaxRadius);
  const int64_t smem = ccvpe_pose_hypotheses_smem_bytes(H, W);
  CCVPE_REQUIRE(smem > 0, "ccvpe_pose_hypotheses: a %dx%d map's band of %d rows does not fit one CTA's shared memory "
                "(%lld bytes at most)", H, W, (H + kHypCtas - 1) / kHypCtas, (long long)kHypSmemMax);
  const uintptr_t a4 = (uintptr_t)heatmap | (uintptr_t)ori | (uintptr_t)rc | (uintptr_t)value | (uintptr_t)mass |
                       (uintptr_t)cs | (uintptr_t)count;
  CCVPE_REQUIRE((a4 & 3u) == 0 && (((uintptr_t)idx | (uintptr_t)angle_deg) & 7u) == 0,
                "ccvpe_pose_hypotheses: misaligned pointer");
  static thread_local uint64_t attr = 0;
  if (first_use_on_device(attr))   // a failure here surfaces as the launch's error
    cudaFuncSetAttribute(pose_hypotheses_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHypSmemMax);
  cudaStream_t st = (cudaStream_t)stream;
  pose_hypotheses_kernel<<<dim3(kHypCtas, B), kHypThreads, (size_t)smem, st>>>(heatmap, ori, H, W, k, radius, idx, rc,
                                                                               value, mass, cs, angle_deg, valid, count);
  CCVPE_LAUNCH_CHECK("pose_hypotheses_kernel");
  return CCVPE_OK;
}
