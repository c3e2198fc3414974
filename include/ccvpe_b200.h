/*
 * ccvpe_b200.h -- C ABI of libccvpe_b200.so: the post-encoder hot path of tudelft-iv/CCVPE as sm_100a CUDA kernels.
 *
 * The reference has no FFI layer (it is pure Python/PyTorch); its only boundary for this path is
 * `CVM_*.forward(grd, sat)` in models.py.  The entry points below are the operators that boundary decomposes into
 * (SURVEY.md section 8(a), rows a1..a13); `ccvpe_b200/models.py` re-assembles them behind the reference's own
 * forward signatures.  Each function cites the reference lines it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; nothing here allocates, frees or
 *     synchronises: outputs and scratch are caller-allocated, work is enqueued on `stream` (a cudaStream_t).
 *   - return value: 0 = ok; <0 = error (CCVPE_ERR_*); `ccvpe_last_error()` returns a thread-local message.
 *   - activations are channels-last ("NHWC": [B, H, W, C], C contiguous) with element type `dtype`
 *     (CCVPE_F32 or CCVPE_BF16); accumulation is always fp32.  Tensors returned to the caller of
 *     `forward` (scores, logits, heatmap, orientation field) are fp32 in the reference's NCHW layout.
 *   - all channel counts must be multiples of 8 (true for every layer of the four reference models).
 */
#ifndef CCVPE_B200_H_
#define CCVPE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCVPE_ABI_VERSION 3

enum { CCVPE_F32 = 0, CCVPE_BF16 = 1 };

enum {
  CCVPE_OK = 0,
  CCVPE_ERR_BAD_ARGUMENT = -1,  /* null pointer, negative size, misaligned pointer ...            */
  CCVPE_ERR_UNSUPPORTED = -2,   /* shape / dtype / backend combination not implemented            */
  CCVPE_ERR_CUDA = -3,          /* a CUDA runtime / driver call or kernel launch failed           */
  CCVPE_ERR_NO_DEVICE = -4      /* no sm_100 device visible                                        */
};

/* backends for the dense contractions */
enum {
  CCVPE_BACKEND_AUTO = 0,    /* tcgen05 when dtype == BF16 and the shape is supported, else SIMT  */
  CCVPE_BACKEND_SIMT = 1,    /* fp32-accumulate CUDA-core implicit GEMM (any dtype) -- the fp32 parity path */
  CCVPE_BACKEND_TCGEN05 = 2  /* TMA-fed tcgen05.mma tiles, accumulators in TMEM (bf16 operands)   */
};

int ccvpe_abi_version(void);
const char* ccvpe_last_error(void);
/* number of kernels this library has launched (all threads of the process) since the last reset */
int64_t ccvpe_launch_count(void);
void ccvpe_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------------------------
 * a1  Ground descriptor heads -- reference models.py:22-31, 57-97, 152-157 (and :355-395, :662-699, :961-998).
 *   g[b, w*c + ch] = sum_h v[h] * (sum_k W[ch,k] * F[b,k,h,w] + bias1[ch]) + bias2
 * feat: ground feature volume, logical [B, K, H, W] addressed through element strides (sb, sk, sh, sw) so both
 *       NCHW and channels-last encoder outputs are accepted.  w1 [c, K] fp32, b1 [c] fp32, w2 [H] fp32, b2 [1] fp32.
 * out : fp32 [B, W*c].  scratch: fp32, at least B*K*W elements.
 * ------------------------------------------------------------------------------------------------------------- */
int ccvpe_grd_descriptor(const void* feat, int dtype, int B, int K, int H, int W,
                         int64_t sb, int64_t sk, int64_t sh, int64_t sw,
                         const float* w1, const float* b1, const float* w2, const float* b2, int c,
                         float* out, float* scratch, void* stream);

/* All heads of a model in two launches (the feature volume is read once): HOST arrays of n_heads (<= 6) device
 * pointers / channel counts; out[l] fp32 [B, W*c[l]]; scratch fp32 >= n_heads*B*K*W elements; K % 4 == 0. */
int ccvpe_grd_descriptors(const void* feat, int dtype, int B, int K, int H, int W,
                          int64_t sb, int64_t sk, int64_t sh, int64_t sw, int n_heads,
                          const float* const* w1, const float* const* b1, const float* const* w2, const float* const* b2,
                          const int32_t* c, float* const* out, float* scratch, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Generic implicit GEMM used for a3 (aerial cell descriptors), a8 (ConvTranspose2d k2 s2) and a9 (3x3 convs):
 *
 *   acc[m, n] = sum_{tap=(ty,tx)} sum_{src in {0,1}} sum_{k < c_src}
 *                   A_src[b, ho*stride + ty - pad, wo*stride + tx - pad, k] * Wt[tap][koff_src + k][n]
 *   y[m, n]   = act( acc[m, n] * row_scale[m] + row_r1[m] * r1_w[n] + bias[n] )          m = (b, ho, wo)
 *
 * Two channels-last sources are K-concatenated on the fly: this is how torch.cat([x, skip]) (models.py:208, 230, ...)
 * and torch.cat([max, normalize(x)]) (models.py:205, 228, ...) are executed without materialising the concat:
 *   row_scale = 1/max(||x_m||, 1e-12)  (F.normalize, models.py:33-40), row_r1 = max-over-rolls score, r1_w = W[0, :].
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct ccvpe_igemm_desc {
  /* sources (a1 may be NULL with c1 == 0); both have spatial size [B, Hin, Win]; ld* = channel stride in elements
   * of one pixel (>= c*, lets a source be a channel-slice of a wider tensor) */
  const void* a0; const void* a1;
  int32_t c0, c1, ld0, ld1;
  int32_t B, Hin, Win, Hout, Wout;
  int32_t stride, kh, kw, pad;
  int32_t N;                     /* GEMM N: Cout, or 4*Cout ordered (i, j, co) for the k2 s2 transposed conv        */
  int32_t dtype;                 /* CCVPE_F32 / CCVPE_BF16: element type of sources and weights                     */
  /* weights, one of (depending on backend):
   *   w_kn : [taps][c0 + c1][N]                     (N contiguous)       -- SIMT backend
   *   w_nk : [N][taps][pad(c0) + pad(c1)]           (K contiguous, bf16) -- tcgen05 backend; pad(c) rounds c up to
   *          a multiple of the source's K-block width kw(c) = 16 if c <= 16, 32 if c <= 32, else 64 (zero filled)  */
  const void* w_kn; const void* w_nk;
  const float* bias;             /* [N] fp32 or NULL                                                                */
  const float* row_scale;        /* [M] fp32 or NULL                                                                */
  const float* row_r1;           /* [M] fp32 or NULL                                                                */
  const float* r1_w;             /* [N] fp32 (required iff row_r1)                                                  */
  int32_t relu;
  /* output */
  int32_t out_mode;              /* 0: channels-last [M, ldo]; 1: pixel-shuffle of a k2 s2 transposed conv into
                                    channels-last [B, 2*Hout, 2*Wout, ldo]; 2: fp32 planar NCHW [B, N, Hout, Wout]  */
  int32_t out_dtype;             /* CCVPE_F32 / CCVPE_BF16 (mode 2 requires F32)                                    */
  int32_t ldo;                   /* channel stride of the output pixel (modes 0/1)                                  */
  void* out;
  int32_t backend;               /* CCVPE_BACKEND_*                                                                 */
} ccvpe_igemm_desc;

/* a3: models.py:102-104,173-184 | a8: models.py:109-124,207,229,... | a9: models.py:42-47,110-127,209,231,...     */
int ccvpe_igemm(const ccvpe_igemm_desc* desc, void* stream);
/* which kernel ccvpe_igemm would launch for this descriptor: 0 = igemm_simt_kernel, 1 = igemm_tcgen05_kernel,
 * 2 = conv_ring_tcgen05_kernel; < 0 = error.  (Used by the benchmark to attribute time to kernels.) */
int ccvpe_igemm_plan(const ccvpe_igemm_desc* desc);

/* ---------------------------------------------------------------------------------------------------------------
 * a4 a5 a6  Rolled cosine matching of one decoder level -- reference models.py:186-202 (x6 levels), prior-limited
 * variant :489-511, KITTI :788-920, Oxford centred window :1094.
 *
 *   window_i[k]   = x[(k + offset + shift_i) mod C]          k = 0..L-1,  shift_i = roll_index_i * roll_stride
 *   scores[b,i,p] = sum_k g[b,k] * window_i[k,p] / ( sqrt(sum_k window_i[k,p]^2) * sqrt(sum_k g[b,k]^2) )
 *   max[b,p]      = max over the rolls i with bit i set in max_mask
 *   inv_norm[b,p] = 1 / max( sqrt(sum_c x[b,p,c]^2), 1e-12 )                  (the F.normalize of models.py:205)
 *
 * x: channels-last [B, HW, C] (dtype).  g: fp32 [B, L].  shifts: HOST array of n_rolls ints (any sign).
 * Outputs (any may be NULL): scores fp32 [B, n_rolls, HW] (the reference's NCHW score volume),
 *   scores_cl (dtype) [B, HW, ld_scores_cl] channels-last copy (pad channels zero; feeds the orientation decoder,
 *   models.py:323), max fp32 [B, HW], inv_norm fp32 [B, HW], xhat (dtype) [B, HW, C] = normalised map.
 * scratch: fp32, at least ccvpe_match_scratch_elems(B, C, n_rolls) elements.
 * ------------------------------------------------------------------------------------------------------------- */
int64_t ccvpe_match_scratch_elems(int B, int C, int n_rolls);
/* which kernel ccvpe_match_level would launch: 0 = match_level_simt_kernel (fp32 inputs, CCVPE_BACKEND_SIMT),
 * 1 = match_tcgen05_kernel (bf16: full-circle and windowed levels); < 0 = error. */
int ccvpe_match_plan(int dtype, int C, int L, int offset, const int32_t* shifts_host, int n_rolls, int ld_scores_cl,
                     int backend);
int ccvpe_match_level(const void* x, int dtype, int B, int HW, int C,
                      const float* g, int L, int offset, const int32_t* shifts_host, int n_rolls, uint32_t max_mask,
                      float* scores, void* scores_cl, int ld_scores_cl, float* max_out, float* inv_norm, void* xhat,
                      float* scratch, int backend, void* stream);

/* a10  softmax over the flattened heatmap logits -- reference models.py:319-320.
 * logits fp32 [B, n]; heatmap fp32 [B, n]; scratch fp32 >= ccvpe_softmax_scratch_elems(B, n). */
int64_t ccvpe_softmax_scratch_elems(int B, int64_t n);
int ccvpe_softmax_heatmap(const float* logits, float* heatmap, int B, int64_t n, float* scratch, void* stream);

/* a12  orientation vector-field normalisation -- reference models.py:341 (F.normalize p=2 dim=1, eps 1e-12).
 * in: channels-last [B, HW, ld] (dtype), first 2 channels = (cos, sin); out: fp32 planar [B, 2, HW]. */
int ccvpe_ori_normalize(const void* in, int dtype, int ld, float* out, int B, int64_t HW, void* stream);

/* a13  argmax pose decode -- reference train_VIGOR.py:290-326 (+ 8 copies in the other scripts).
 * heatmap fp32 [B, H*W]; ori fp32 planar [B, 2, H*W].
 * idx[b]   = first index of the maximum of heatmap[b] (numpy argmax semantics; a NaN counts as the maximum)
 * rc[b]    = (idx / W, idx % W);  cs[b] = (ori[b,0,idx], ori[b,1,idx])
 * valid[b] = |cos| <= 1 && |sin| <= 1;  angle_deg[b] = valid ? (sin < 0 ? fmod(degrees(-acos(cos)), 360) (python %)
 *            : degrees(acos(cos))) : NaN,   evaluated in float64.
 * scratch: >= ccvpe_pose_scratch_bytes(B, H*W) bytes. */
int64_t ccvpe_pose_scratch_bytes(int B, int64_t n);
int ccvpe_pose_decode(const float* heatmap, const float* ori, int B, int H, int W,
                      int64_t* idx, int32_t* rc, float* cs, double* angle_deg, uint8_t* valid,
                      void* scratch, void* stream);

/* a13  pose hypotheses -- the k strongest mutually exclusive location modes of each heatmap, in one launch.
 * heatmap fp32 [B, H*W]; ori fp32 planar [B, 2, H*W]; 1 <= k <= 64; 0 <= radius <= 32767.  For each pair:
 *   candidates: the pixels whose value is >= every in-bounds 8-neighbour (fixed from the original map), ordered by value,
 *     highest first, ties to the smaller flat index i*W + j (NumPy's first occurrence; -0 and +0 are equal values);
 *   greedy claim: the first candidate not yet claimed becomes the next hypothesis and claims every pixel of its disc
 *     (i - i0)^2 + (j - j0)^2 <= radius^2 (integer arithmetic); stop after k hypotheses or when the candidates run out.
 * Hypothesis t < count[b], at slot [b, t]:
 *   idx = i0*W + j0;  rc = (i0, j0);  value = heatmap[b, idx];
 *   mass = the sum of the heatmap over the pixels of its disc that no earlier hypothesis claimed, accumulated in float64
 *     in a fixed order and rounded once to float32 (the masses partition the claimed probability: their sum is <= 1 for a
 *     softmax heatmap);
 *   cs, angle_deg, valid: ccvpe_pose_decode's rule at idx.
 * Slots t >= count[b]: idx = -1, rc = (-1, -1), value = mass = cs = angle_deg = NaN, valid = 0.
 * A heatmap holding any NaN has no neighbourhood order: count = 0.  +-inf compare as ordinary values (an all -inf map
 * gives idx 0, as ccvpe_pose_decode).  With k = 1 idx, rc, cs, angle_deg and valid equal ccvpe_pose_decode's on every
 * NaN-free map (its first-occurrence maximum is always a mode).
 * Outputs: idx [B, k], rc [B, k, 2], value / mass [B, k], cs [B, k, 2], angle_deg [B, k], valid [B, k], count [B], each
 * naturally aligned.  One 8-CTA cluster per pair holds the map in shared memory, a band of ceil(H/8) rows (+ 2 halo rows)
 * per CTA: ccvpe_pose_hypotheses_smem_bytes(H, W) is that per-CTA need, or -1 where it does not fit (a 512x512 map needs
 * 143 376 bytes); such maps, like every other bad argument, are refused with CCVPE_ERR_BAD_ARGUMENT before any launch.
 * Reads the heatmap once; no workspace, no allocation, no synchronisation; deterministic; graph-capturable. */
int64_t ccvpe_pose_hypotheses_smem_bytes(int H, int W);
int ccvpe_pose_hypotheses(const float* heatmap, const float* ori, int B, int H, int W, int k, int radius,
                          int64_t* idx, int32_t* rc, float* value, float* mass, float* cs, double* angle_deg,
                          uint8_t* valid, int32_t* count, void* stream);

/* Sequential location filter -- one Bayes-filter step per frame, fusing each heatmap with the motion-propagated belief of
 * the previous frame.  belief fp32 [B, H*W] (updated in place: one location distribution per track, on the pixel grid of
 * the track's current aerial crop); heatmap fp32 [B, H*W] (this frame's model output, must not overlap belief); motion
 * float64 [B, 6] on the device, read when the kernels run (a captured step replays with whatever it then holds);
 * 0 <= sigma <= 32 (pixels); 0 <= epsilon <= 1; 1 <= B <= 65535; 1 <= H, W <= 4096.  Per track:
 *   1. predict: motion a[0..5] maps a pixel centre of the new grid to a coordinate of the previous one (the convention of
 *      ccvpe_affine_u8 / Pillow's AFFINE data).  For new pixel (i, j), in float64 with every operation rounded:
 *        u = ((a0*(j+0.5) + a1*(i+0.5)) + a2) - 0.5,   v = ((a3*(j+0.5) + a4*(i+0.5)) + a5) - 0.5;
 *      p = |a0*a4 - a1*a3| * bilinear(old belief at (v, u)) with the weights of (u - floor u, v - floor v), each tap outside
 *      the grid contributing 0 (zero padding: probability leaving the crop is lost); a coordinate whose 4 taps all lie
 *      outside (NaN, inf or huge ones included) gives p = 0;
 *   2. process noise: p convolved with the separable Gaussian w_d ~ exp(-d^2 / (2 sigma^2)), |d| <= r = ceil(3 sigma),
 *      normalised to sum 1 (float64, rounded to float32), zero padded; rows first, then columns; sigma = 0 is the identity;
 *   3. mix: prior = (1 - epsilon) * p + epsilon / (H*W)   (float64, no renormalisation first);
 *   4. update: q = prior * heatmap (float64), Z = sum q in float64 in a fixed order; evidence[b] = Z.
 *      Z > 0 and finite: belief = q / Z (q rounded to float32 first), reset[b] = 0;
 *      otherwise (disjoint supports with epsilon = 0, a NaN or inf in the heatmap, a NaN belief): belief = a bitwise copy
 *      of the heatmap, reset[b] = 1.
 * Each blur output is w_0 s_j + sum_{d=1..r} w_d (s_{j-d} + s_{j+d}), accumulated in float32 in that order.  Where q is
 * below float32's normal range, its rounding is absolute (2^-150 / Z in the belief).  Values of prior * heatmap beyond float32's
 * range are not supported.  scratch: >= ccvpe_track_scratch_bytes(B, H, W) bytes (-1 for a refused shape), 8-byte
 * aligned.  belief and heatmap 4-byte, motion and evidence 8-byte aligned.  Every bad argument is refused with
 * CCVPE_ERR_BAD_ARGUMENT before any launch.  Three launches, no allocation, no host synchronisation or copy;
 * deterministic; graph-capturable. */
int64_t ccvpe_track_scratch_bytes(int B, int H, int W);
int ccvpe_track_step(float* belief, const float* heatmap, const double* motion, int B, int H, int W, float sigma,
                     float epsilon, double* evidence, uint8_t* reset, void* scratch, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Encoder glue (SURVEY section 8(f)-2, first step; the encoders themselves stay cuDNN/cuBLAS through PyTorch):
 *   y[b,h,w,c] = SiLU(x[b,h,w,c] + bias[c]);   chan_sum[b,c] += sum_{h,w} y[b,h,w,c]   (optional, caller zeroes it)
 * chan_sum is 64-bit FIXED POINT in units of 2^-20 (CCVPE_SE_SUM_SCALE): integer accumulation is order independent, so
 * the squeeze-excite statistics -- and with them the whole bf16 path -- are bit-reproducible from run to run.
 * x: contiguous channels-last bf16 [B,H,W,C]; bias: bf16 [C] or NULL; y: bf16 with element strides (y_sb, y_sh, y_sw)
 * between images / rows / pixels (channels contiguous) -- e.g. the interior of a padded buffer.  C % 8 == 0.
 * Replaces x*sigmoid(x) after BN (reference efficientnet_pytorch/model.py:105-110) plus F.adaptive_avg_pool2d (:114).
 * ------------------------------------------------------------------------------------------------------------- */
#define CCVPE_SE_SUM_SCALE 1048576.0
int ccvpe_bias_silu_nhwc(const void* x, const void* bias, void* y, int64_t y_sb, int64_t y_sh, int64_t y_sw,
                         int B, int H, int W, int C, int64_t* chan_sum, void* stream);

/* Depthwise KxK conv (K in {3,5}, stride S in {1,2}) over a PRE-PADDED channels-last bf16 buffer, fused with bias, SiLU
 * and the squeeze-excite channel sums (reference efficientnet_pytorch/model.py:108-114 in eval mode, BN folded):
 *   y[b,ho,wo,c] = SiLU(sum_{ky,kx} x[b, ho*S+ky, wo*S+kx, c] * w[ky,kx,c] + bias[c]);  chan_sum[b,c] += sum_{ho,wo} y
 * x: bf16, logical padded size [B,Hp,Wp,C] with element strides (x_sb, x_sh, x_sw), channels contiguous;
 * w: bf16 [K*K, C]; bias: bf16 [C]; y: contiguous bf16 [B,Ho,Wo,C], Ho=(Hp-K)/S+1, Wo=(Wp-K)/S+1; chan_sum int64 fixed point
 * (see ccvpe_bias_silu_nhwc) [B, C] or NULL. */
int ccvpe_dwconv_bias_silu_nhwc(const void* x, int64_t x_sb, int64_t x_sh, int64_t x_sw, int Hp, int Wp,
                                const void* w, const void* bias, void* y, int B, int C, int K, int S,
                                int64_t* chan_sum, void* stream);
/* which kernel ccvpe_dwconv_bias_silu_nhwc would launch for this layer (the launch makes the same choice):
 * 0 = dwconv_bias_silu_kernel, 1 = dwconv_tile_kernel; < 0 = error. */
int ccvpe_dwconv_plan(int B, int C, int Hp, int Wp, int K, int S);

/* Encoder stem (reference efficientnet_pytorch/model.py:296-297 in eval mode, BN folded; circular variant: the reference's
 * models.py circular-padding patch of the ground encoder): 3x3 stride-2 conv over the fp32 NCHW image with the reference's
 * static "same" padding (in_pad_lo / in_pad_hi zero rows and columns before / after the image; circular != 0 wraps the
 * width instead of zero-filling it), + bias + SiLU:
 *   out[b, ho + out_pad_lo, wo + out_pad_lo, co] = SiLU(bias[co] + sum_{ci,ky,kx} x[b,ci,2ho+ky-in_pad_lo,2wo+kx-in_pad_lo] * w[(ci,ky,kx), co])
 * x: fp32 [B,3,H,W]; w: fp32 [27][CO] ordered (ci, ky, kx); bias fp32 [CO]; CO == 32;
 * out: bf16 [B, Ho+out_pad_lo+out_pad_hi, Wo+out_pad_lo+out_pad_hi, CO], Ho = (H+in_pad_lo+in_pad_hi-3)/2+1 (Wo alike); the interior is
 * written, and for circular != 0 also the wrap columns (the zero rows above / below are left untouched). */
int ccvpe_stem_conv_silu_nhwc(const float* x, int B, int H, int W, const float* w, const float* bias, int CO,
                              void* out, int in_pad_lo, int in_pad_hi, int out_pad_lo, int out_pad_hi, int circular,
                              void* stream);

/* The same stem with the f4 input pipeline fused into its loads: x is the uint8 image batch NCHW [B, 3, H, Wsrc]; every load
 * applies ToTensor + Normalize ((u8 / 255 - mean[c]) / std[c], evaluated as one FMA), the per-image panorama roll
 * (torch.roll by shift[b] columns; shift NULL = none) and the limited-FoV crop to the first crop_w columns
 * (reference train_VIGOR.py:55-70, 272-273; datasets.py:118).  mean_host / std_host: HOST float[3]. */
int ccvpe_stem_conv_silu_u8_nhwc(const uint8_t* x, int B, int H, int Wsrc, int crop_w, const int32_t* shift,
                                 const float* mean_host, const float* std_host, const float* w, const float* bias, int CO,
                                 void* out, int in_pad_lo, int in_pad_hi, int out_pad_lo, int out_pad_hi, int circular,
                                 void* stream);

/* Circular width padding of a padded channels-last bf16 image [B, H+lo+hi, W+lo+hi, C] (pad the same on both axes, as
 * the depthwise convs use it) whose interior is already written: the lo left / hi right padding columns of the interior
 * rows receive the wrapped-around interior columns (the reference's circular-padding patch of the ground encoder,
 * models.py: F.pad(..., mode='circular') along the width).  The zero rows above / below are left untouched.  C % 8 == 0. */
int ccvpe_wrap_columns_nhwc(void* buf, int B, int H, int W, int C, int pad_lo, int pad_hi, void* stream);

/* Squeeze-excite gate folded into the projection weights (reference efficientnet_pytorch/model.py:113-121 in eval mode):
 *   mean = chan_sum / CCVPE_SE_SUM_SCALE * inv_hw;  h = SiLU(w_red mean + b_red);  g = sigmoid(w_se h + b_se);  wg[b] = w_proj * diag(g[b])
 * chan_sum int64 fixed point [B, mid] (from ccvpe_dwconv_bias_silu_nhwc); w_red bf16 [R, mid]; b_red bf16 [R]; w_se bf16 [R, mid]
 * (the excite weights TRANSPOSED, so the gate mat-vec reads them coalesced); b_se bf16 [mid]; w_proj bf16 [cout, mid]; wg bf16 [B, cout, mid] = the per-image B operand of the projection GEMM
 * (W (g . x) == (W diag(g)) x, so the broadcast multiply over the expanded activation never happens).  mid % 8 == 0.
 * rep > 1: wg is bf16 [B, rep*cout, rep*mid], block diagonal with rep copies of wg[b] -- the weights of `rep` consecutive
 * pixels packed into one GEMM row (ccvpe_mbconv_project_nhwc on [B, HW/rep, rep*mid]).  gate_ws: fp32 [B, mid] workspace or
 * NULL; required for rep > 1, and when given the deep blocks run as two launches (gate, then a flat scaling pass). */
int ccvpe_se_gate_scale(const int64_t* chan_sum, float inv_hw, const void* w_red, const void* b_red, const void* w_se,
                        const void* b_se, const void* w_proj, void* wg, int B, int mid, int R, int cout, int rep,
                        float* gate_ws, void* stream);

/* Pointwise (1x1) convolution + bias + SiLU over channels-last bf16 pixels on the tcgen05 pipeline -- the MBConv expand
 * step and the encoder head (reference efficientnet_pytorch/model.py:100-106, 312-314 in eval mode, BN folded):
 *   out[b, h + pad_lo, w + pad_lo, n] = SiLU(sum_k x[(b,h,w), k] * w_nk[n, k] + bias[n])
 * x: bf16 [B*H*W, K] with row stride ldx (elements); w_nk: bf16 [N][pad(K)] in the K-block padded layout documented for
 * ccvpe_igemm_desc.w_nk; bias fp32 [N] or NULL; out: bf16 image [B, H+pad_lo+pad_hi, W+pad_lo+pad_hi, N] whose interior is
 * written (the border is left untouched: the depthwise convolution's zero padding lives there).  K % 8 == N % 8 == 0. */
int ccvpe_pointwise_silu_nhwc(const void* x, int B, int H, int W, int K, int ldx, const void* w_nk, const float* bias,
                              int N, void* out, int pad_lo, int pad_hi, void* stream);

/* f2  MBConv projection -- reference efficientnet_pytorch/model.py:115-131 (squeeze-excite multiply, _project_conv + _bn2,
 * identity skip), batched over images because the gate is folded into PER-IMAGE weights wg = W_proj . diag(gate[b])
 * (ccvpe_se_gate_scale):
 *   out[b, p, n] = sum_k d[b, p, k] * wg[b, n, k]  (+ residual[b, p, n])          fp32 accumulation, rounded once to bf16
 *   out_biased[b, p, n] = bf16(out[b, p, n]) + bias[n]                              (optional; the decoder's skip tensor)
 * d: bf16 [B, HW, mid]; wg: bf16 [B, cout, mid]; residual: bf16 [B, HW, cout] or NULL; bias: bf16 [cout] (required iff
 * out_biased); out / out_biased: bf16 [B, HW, cout].  mid % 8 == cout % 8 == 0; all pointers 16-byte aligned. */
int ccvpe_mbconv_project_nhwc(const void* d, const void* wg, const void* residual, const void* bias, void* out,
                              void* out_biased, int B, int HW, int mid, int cout, void* stream);

/* f4  Input pipeline after image decoding -- reference train_VIGOR.py:55-70 (ToTensor + Normalize), datasets.py:118
 * (random panorama roll: torch.roll(grd, shift, dims=2)), train_VIGOR.py:272-273 (limited-FoV crop of the panorama):
 *   dst[b, c, h, w] = (src[b, c, h, (w - shift[b]) mod W] / 255 - mean[c]) / std[c]        for w < crop_w
 * src: uint8 image batch, NCHW [B,3,H,W] (nhwc == 0) or NHWC [B,H,W,3] (nhwc != 0); shift: device int32 [B] or NULL;
 * mean_host / std_host: HOST float[3]; dst: fp32 NCHW [B,3,H,crop_w].  Bit-identical to torchvision's transforms. */
int ccvpe_ingest_u8(const uint8_t* src, int nhwc, int B, int H, int W, int crop_w, const int32_t* shift,
                    const float* mean_host, const float* std_host, float* dst, void* stream);

/* f4  Resize before ingest -- reference transforms.Resize([out_h, out_w]) on each image as a PIL image (train_VIGOR.py:55-70),
 * i.e. Pillow's Image.resize((out_w, out_h), BILINEAR) in 8 bits per channel: per axis, integer weights (2^22 fixed point)
 * from Pillow's double-precision coefficient tables, horizontal pass first into a uint8 intermediate, then the vertical pass.
 * Bit-identical to Pillow for any ratio in either direction (downscales by up to 1000x per axis; a factor so large that
 * one output pixel's coefficient tables and uint8 intermediate column do not fit in shared memory is refused with
 * CCVPE_ERR_BAD_ARGUMENT).  src: uint8 image batch, NCHW [B,3,H,W] (nhwc == 0) or NHWC [B,H,W,3] (nhwc != 0);
 * dst: uint8 NCHW [B,3,out_h,out_w] (the layout ccvpe_ingest_u8 and ccvpe_stem_conv_silu_u8_nhwc read), not overlapping src.
 * One launch; the coefficients are computed on the device: no workspace, no allocation, no synchronisation. */
int ccvpe_resize_u8(const uint8_t* src, int nhwc, int B, int H, int W, int out_h, int out_w, uint8_t* dst, void* stream);

/* f4  Geometric augmentation (rotation, shift, scale, shear, crop) -- Pillow's Image.transform(size, AFFINE, a, BILINEAR,
 * fillcolor) in 8 bits per channel, bit-identical; Image.rotate(angle, BILINEAR, center, translate, fillcolor) is such a
 * transform of the matrix it builds.  matrices: DEVICE float64 [B][6], one `a` per image, mapping output pixel centres to
 * input coordinates (read at run time: a captured launch can be replayed with the matrices rewritten in place).
 * dst[b, :, y, x] is pixel (x + left, y + top) of image b's transform, so with left, top >= 0 the output equals
 * Image.transform((left + out_w, top + out_h), ...).crop((left, top, left + out_w, top + out_h)).  Pixels whose source
 * coordinate falls outside the image take fill_host[0..2] (HOST uint8[3], RGB).  src: uint8 NCHW [B,3,H,W] (nhwc == 0)
 * or NHWC [B,H,W,3] (nhwc != 0); dst: uint8 NCHW [B,3,out_h,out_w], not overlapping src.  One launch: no workspace, no
 * allocation, no synchronisation.  Pillow's NEAREST and BICUBIC affine resamplers are not provided. */
int ccvpe_affine_u8(const uint8_t* src, int nhwc, int B, int H, int W, const double* matrices, int out_h, int out_w,
                    int left, int top, const uint8_t* fill_host, uint8_t* dst, void* stream);

/* =================================================================================================================
 * Training step (BASELINE.json configs[4]; reference train_VIGOR.py:120-150, losses.py:4-29): backward kernels.
 * The data gradient of every convolution is a `ccvpe_igemm` call on re-laid-out weights (a 3x3 pad-1 conv's is a 3x3 pad-1
 * conv with flipped, transposed weights; a k2 s2 transposed conv's is a k2 s2 conv and vice versa); what follows are the
 * operators that have no forward counterpart.  All reductions are deterministic (workspace partials, fixed order).
 * ================================================================================================================= */

/* Weight gradient of the implicit GEMM of ccvpe_igemm:
 *   out[tap][c][n] = sum_m A_src[b, ho*stride + ty - pad, wo*stride + tx - pad, c] * G[m, n] * (g_row_scale ? g_row_scale[m] : 1)
 * A sources as in ccvpe_igemm_desc (channels-last, two K-concatenated sources); G: channels-last [B*Hout*Wout, N] with row
 * stride ldg.  3x3 conv: A = layer input, G = dY.  k2 s2 transposed conv: A = dY (the pixel-shuffled output gradient,
 * kh = kw = 2, stride 2), G = the layer input with g_row_scale = 1/||x|| (F.normalize).  k2 s2 cell conv: A = aerial
 * features, G = d(cell descriptors).  out is fp32 in the w_kn layout of the forward weights [taps][c0 + c1][N].
 * Channel counts and strides: multiples of 4.  workspace: >= ccvpe_wgrad_workspace_elems(desc) floats. */
typedef struct ccvpe_wgrad_desc {
  const void* a0; const void* a1;
  int32_t c0, c1, ld0, ld1;
  int32_t B, Hin, Win, Hout, Wout;
  int32_t stride, kh, kw, pad;
  const void* g; int32_t N, ldg;
  const float* g_row_scale;
  int32_t dtype;                 /* CCVPE_F32 / CCVPE_BF16: element type of a0, a1 and g */
  float* out;
  float* workspace; int64_t workspace_elems;
  int32_t backend;               /* CCVPE_BACKEND_* */
} ccvpe_wgrad_desc;
int64_t ccvpe_wgrad_workspace_elems(const ccvpe_wgrad_desc* desc);
int ccvpe_wgrad(const ccvpe_wgrad_desc* desc, void* stream);
/* 0 = wgrad_simt_kernel, 1 = wgrad_tcgen05_kernel; < 0 = error */
int ccvpe_wgrad_plan(const ccvpe_wgrad_desc* desc);

/* Bucketed, weighted column sums over a channels-last image x [B, H, W, ld] (first C channels):
 *   out[(y % s) * s + (x % s)][c] = sum_{b,y,x} w[b, y/s, x/s] * x[b, y, x, c]        (w NULL: 1;  s = 1 or 2)
 * s = 1: bias gradient of a conv.  s = 2, w = max-score map: gradient of the rank-1 weight row of a k2 s2 transposed conv
 * (torch.cat([max, normalize(x)]) channel 0, models.py:205); s = 2, w NULL: the four bucket sums of its bias gradient.
 * out fp32 [s*s][C]; workspace >= ccvpe_colsum_workspace_elems(B*H*W, C, s) floats. */
int64_t ccvpe_colsum_workspace_elems(int64_t n_pix, int C, int s);
int ccvpe_colsum(const void* x, int dtype, int B, int H, int W, int C, int ld, const float* w, int s, float* out,
                 float* workspace, void* stream);

/* y[m, :] = x[m, :] * scale[m] over a channels-last matrix [M, C] (C % 4 == 0): the L2-normalised aerial map as an explicit
 * tensor (models.py:205), the G operand of the tensor-core weight gradient of the transposed convs. */
int ccvpe_scale_rows(const void* x, int dtype, const float* scale, void* y, int64_t M, int C, void* stream);
/* ReLU backward in place: dh[i] = h[i] > 0 ? dh[i] : 0 (models.py:45).  n % 4 == 0. */
int ccvpe_relu_bwd(void* dh, const void* h, int dtype, int64_t n, void* stream);
/* planar fp32 [B, N, HW] -> channels-last (dtype) [B, HW, ld], channels >= N zero filled (incoming d logits) */
int ccvpe_planar_to_cl(const float* src, void* dst, int dtype, int B, int N, int64_t HW, int ld, void* stream);
/* channels-last (dtype) [B, HW, ld] (first N channels) -> planar fp32 [B, N, HW] (outgoing gradients of NCHW inputs) */
int ccvpe_cl_to_planar(const void* src, int dtype, float* dst, int B, int N, int64_t HW, int ld, void* stream);
/* Backward of the orientation-field normalisation (models.py:341): v channels-last [B, HW, ldv] (raw 2-vector field),
 * d_ori planar fp32 [B, 2, HW] -> dv channels-last (dv_dtype) [B, HW, ldo], channels >= 2 zero filled. */
int ccvpe_ori_normalize_bwd(const void* v, int v_dtype, int ldv, const float* d_ori, void* dv, int dv_dtype, int ldo,
                            int B, int64_t HW, void* stream);

/* Backward of one matching level (models.py:186-205): given the saved forward scores, the incoming gradients of the score
 * volume (d_scores fp32 [B, R, HW] and/or d_scores_cl: columns 0..R-1 of a (dtype) [B*HW, ld_dscl] matrix -- the
 * orientation decoder's input gradient at the bottleneck level; either may be NULL), of the max-over-orientations channel
 * (d_max: column 0 of a (dtype) [B*HW, ld_dmax] matrix, may be NULL) and of the normalised map (d_xhat / d_xhat2: first C
 * columns of (dtype) [B*HW, ld] matrices, summed; may be NULL) -> dx (dtype) [B, HW, C] and dg fp32 [B, L].
 * scratch: >= ccvpe_match_bwd_scratch_elems floats. */
int64_t ccvpe_match_bwd_scratch_elems(int B, int HW, int C, int n_rolls);
int ccvpe_match_level_bwd(const void* x, int dtype, int B, int HW, int C, const float* g, int L, int offset,
                          const int32_t* shifts_host, int n_rolls, uint32_t max_mask, const float* scores,
                          const float* d_scores, const void* d_scores_cl, int ld_dscl, const void* d_max, int ld_dmax,
                          const void* d_xhat, int ld_dxhat, const void* d_xhat2, int ld_dxhat2, void* dx, float* dg,
                          float* scratch, void* stream);

/* Training losses, value and gradient in one call (reference losses.py).  All tensors fp32; workspace >=
 * ccvpe_loss_workspace_elems(B) floats; `loss` is a device scalar.
 *   infoNCE (losses.py:4-20): scores, labels [B, n]; positives = labels > 1e-2; d_scores [B, n]
 *   cross entropy (losses.py:23-24): logits, labels [B, n]; d_logits [B, n]
 *   orientation (losses.py:28-29): ori, gt_ori planar [B, 2, HW], gt [B, HW]; d_ori [B, 2, HW] */
int64_t ccvpe_loss_workspace_elems(int B);
int ccvpe_infonce_loss(const float* scores, const float* labels, int B, int64_t n, float temperature, float* loss,
                       float* d_scores, float* workspace, void* stream);
int ccvpe_cross_entropy_loss(const float* logits, const float* labels, int B, int64_t n, float* loss, float* d_logits,
                             float* workspace, void* stream);
int ccvpe_orientation_loss(const float* ori, const float* gt_ori, const float* gt, int B, int64_t HW, float* loss,
                           float* d_ori, float* workspace, void* stream);

/* The same losses from compact labels.  A pair's orientation-binned map is rank 1, gt_with_ori[b, r] = gt[b] * bin_w[b, r],
 * and its orientation field is one unit vector, gt_ori[b, :, p] = ori_vec[b, :]; these read the factors instead of the maps
 * and give the same loss and gradient bits as the calls above fed the materialised maps.
 *   label pyramid: gt [B, H, W] (16-byte aligned; H, W multiples of 64, else CCVPE_ERR_BAD_ARGUMENT) -> out, the six
 *     max_pool2d(gt, k, stride=k) maps, k = 64, 32, 16, 8, 4, 2 in this order; level l (k = 64 >> l) is [B, H/k, W/k] at
 *     element offset B * sum_{m<l} (H >> (6-m)) * (W >> (6-m)) (one 64x64 tile per CTA, read once).  NaN propagates.
 *   infoNCE: scores [B, R, HW] of one level, pooled [B, HW] its label pyramid level, bin_w [B, R] (>= 0); the labels are
 *     the correctly rounded products pooled[b, p] * bin_w[b, r].  R * HW < 2^31.  d_scores [B, R, HW].
 *   orientation: ori planar [B, 2, HW], ori_vec [B, 2], gt [B, HW]; d_ori [B, 2, HW]. */
int ccvpe_gt_pyramid(const float* gt, int B, int H, int W, float* out, void* stream);
int ccvpe_infonce_loss_binned(const float* scores, const float* pooled, const float* bin_w, int B, int R, int64_t HW,
                              float temperature, float* loss, float* d_scores, float* workspace, void* stream);
int ccvpe_orientation_loss_const(const float* ori, const float* ori_vec, const float* gt, int B, int64_t HW,
                                 float* loss, float* d_ori, float* workspace, void* stream);

/* The compact labels of a batch of poses, in one launch.  poses: float64 [B, 3], rows (row, col, angle_deg), read when the
 * kernel runs (a captured launch replays with whatever the buffer holds then).  Writes
 *   gt [B, H, W] (16-byte aligned; H, W positive multiples of 64): gt[b, i, j] = float32(exp(-(((i - row)^2 + (j - col)^2)
 *     / (2 * sigma^2)))), evaluated in float64 without contractions and rounded once (NumPy float64's formula); a
 *     non-finite centre gives NaN where NumPy does;
 *   pyramid: ccvpe_gt_pyramid(gt)'s six levels, in its layout;
 *   bin_weights [B, n_bins] and ori_vec [B, 2]: VIGOR's 18-degree rule, bit-identical to losses.orientation_labels
 *     (Python float arithmetic); an angle outside [0, 360) or non-finite gives NaN weights and vector.
 * sigma > 0 and finite, 10 <= n_bins <= 32; otherwise, or on bad sizes or alignment, CCVPE_ERR_BAD_ARGUMENT.  No workspace,
 * no allocation, no synchronisation. */
int ccvpe_pose_labels(const double* poses, int B, int H, int W, double sigma, int n_bins, float* gt, float* pyramid,
                      float* bin_weights, float* ori_vec, void* stream);

/* Backward of the ground descriptor heads (models.py:57-97, 152-157); arguments as ccvpe_grd_descriptors plus the incoming
 * dg[l] fp32 [B, W*c[l]].  Outputs: dfeat fp32 [B, K, H, W] contiguous (NCHW), dw1[l] [c, K], db1[l] [c], dw2[l] [H],
 * db2[l] [1].  scratch: fp32, >= 2*n_heads*B*K*W elements. */
int ccvpe_grd_descriptors_bwd(const void* feat, int dtype, int B, int K, int H, int W, int64_t sb, int64_t sk, int64_t sh,
                              int64_t sw, int n_heads, const float* const* w1, const float* const* b1,
                              const float* const* w2, const int32_t* c, const float* const* dg, float* dfeat,
                              float* const* dw1, float* const* db1, float* const* dw2, float* const* db2, float* scratch,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CCVPE_B200_H_ */
