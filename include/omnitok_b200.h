/*
 * omnitok_b200 -- C ABI of the B200 (sm_100a) kernels behind OmniTokenizer_VQGAN.encode/decode.
 *
 * The reference (FoundationVision/OmniTokenizer) has no FFI of its own: its boundary is the
 * Python module API of OmniTokenizer_VQGAN (OmniTokenizer/omnitokenizer.py:63-413).  Each entry
 * point below replaces one group of torch library calls on that path; the reference call site
 * it stands in for is cited next to it (paths relative to /root/reference/OmniTokenizer/).
 *
 * Conventions
 *   - all pointers are DEVICE pointers owned by the caller (fp32 unless noted); nothing is
 *     allocated or retained; outputs may not alias inputs unless stated.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*).
 *   - return 0 on success, negative on error (OMT_E_*); omt_last_error() gives the message
 *     (thread-local).  There is NO CPU fallback: a non-sm_100 device returns OMT_E_ARCH.
 *   - activations live in ONE canonical layout  X[B][T'][N][C]  (C fastest; identical to the
 *     reference's "(b t) (h w) d" tensor).  "rows" are (b,t',n) triples, M = B*T'*N.
 *   - a "row map" (seg, seg_stride, seg_off) maps logical GEMM row r to physical row
 *     (r / seg) * seg_stride + seg_off + (r % seg); seg <= 0 means identity.  It is how the
 *     first-frame / rest-frames patch matrices address the canonical buffer without a concat.
 */
#ifndef OMNITOK_B200_H_
#define OMNITOK_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OMT_ABI_VERSION 2

#define OMT_OK 0
#define OMT_E_ARG (-1)    /* bad shape / alignment / null pointer */
#define OMT_E_ARCH (-2)   /* device is not sm_100 */
#define OMT_E_CUDA (-3)   /* a CUDA runtime call failed */
#define OMT_E_UNSUPPORTED (-4)

typedef void* omt_stream_t;

int omt_abi_version(void);
const char* omt_last_error(void);
/* sm count / compute capability of the current device */
int omt_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* GEMM epilogue selectors */
#define OMT_EPI_NONE 0
#define OMT_EPI_GEGLU 1   /* packed columns (2j, 2j+1) = (value, gate): C[:, j] = gelu_erf(gate) * value */
#define OMT_EPI_QKV 2     /* dual-A forms: rope + l2norm + scale on the q / k heads (attention.py:417-437) */
#define OMT_EPI_QKV_PLANES 3   /* omt_linear_h: the same, but q / k / v leave as fp16 operand planes for omt_attn_spatial_h */

/* GEMM math selectors */
#define OMT_MATH_FP32 0      /* CUDA-core FFMA, exact fp32 (parity anchor) */
#define OMT_MATH_3XTF32 1    /* tcgen05 kind::tf32, error-compensated hi/lo split, fp32 accumulate in TMEM */
#define OMT_MATH_F16X3 3     /* tcgen05 kind::f16 on pre-split fp16 hi / lo operand planes (omt_linear_h) */

/* C[M, N] = A[M, K] . W[N, K]^T (+ bias[N]) (+ residual[M, N]); nn.Linear everywhere on the path:
 * attention.py:411 (to_q / to_kv), :486 (to_out), :271/:288 (window qkv / proj), :164/:167 (FF),
 * omnitokenizer.py:809,819 (patch embed), :1007,1013 (to_pixels).
 * W must be allocated with rows padded up to a multiple of 128 (zero rows); K % 8 == 0 (fp32 path)
 * or K % 32 == 0 (tcgen05 paths).  With OMT_EPI_GEGLU, N counts packed columns and C has N/2 columns.
 * residual may alias C (same ld): out-of-place is not required.  For OMT_MATH_3XTF32 `W` must be the
 * tf32-rounded (round-to-nearest, low 13 mantissa bits zero) high part of the weight and `W_lo` the
 * exact remainder (same shape); W_lo is ignored (may be NULL) for FP32. */
int omt_linear(const float* A, int lda, int a_seg, int a_seg_stride, int a_seg_off,
               const float* W, const float* W_lo,
               float* C, int ldc, int c_seg, int c_seg_stride, int c_seg_off,
               int M, int N, int K,
               const float* bias, const float* residual, int ldr,
               int epilogue, int math, omt_stream_t stream);

/* Dual-A form: C[:, :n_split] = A1 . W[:n_split]^T and C[:, n_split:] = A2 . W[n_split:]^T in ONE launch.
 * Attention.forward projects q from the LayerNormed input and k, v from the RAW input
 * (attention.py:407-412); stacking [Wq; Wkv] and switching the A tensor map per output tile fuses the two
 * nn.Linear calls without changing either result.  n_split % 256 == 0; same lda for A1 and A2. */
int omt_linear2(const float* A1, const float* A2, int n_split, int lda, const float* W, const float* W_lo,
                float* C, int ldc, int M, int N, int K, int math,
                /* optional fused q/k preparation (what omt_qk_prep does), q_scale == NULL disables it:
                 * columns [0, qk_cols) are heads of 64; the first half carry q (q_scale), the second k (k_scale);
                 * rope tables [tokens, 32] or NULL; the rope position of row m is m % tokens */
                const float* q_scale, const float* k_scale, const float* rope_cos, const float* rope_sin,
                int qk_cols, int tokens, omt_stream_t stream);

/* y[r,:] = (x[r,:] - mean) * rstd * w + b over C channels (C % 4 == 0, C <= 1024); b may be NULL.
 * attention.py:73-80 (LayerNorm, beta buffer), :163 (nn.LayerNorm in FeedForward), :688 (norm_out).
 * x may alias y.  (seg, seg_stride, seg_off) is a row map applied to BOTH x and y (patch embed:
 * the first-frame and rest-frames rows of X carry different LayerNorm weights, omnitokenizer.py:811,821). */
int omt_layernorm(const float* x, int ldx, float* y, int ldy, const float* w, const float* b,
                  int M, int C, float eps, int seg, int seg_stride, int seg_off, omt_stream_t stream);

/* Patch gather + LayerNorm (omnitokenizer.py:806-808 / :814-817: Rearrange + nn.LayerNorm).
 * video (B, Cin, T, H, W) fp32 contiguous.  first=1: frame 0, rows (b,h,w), features (c,p1,p2);
 * first=0: frames 1.., rows (b,t,h,w), features (c,pt,p1,p2).  A is [rows, K] dense.
 * ln_w == ln_b == NULL: plain patch gather (im2col of the strided Conv3d of patch_embed='cnn', omnitokenizer.py:823-838).
 * A_hi != NULL: the rows are written as fp16 hi / lo operand planes [rows, K] instead of A (A may be NULL);
 * A_rs != NULL: in the row-scaled form, inverse row scales to A_rs [rows]. */
int omt_patchify_ln(const float* video, float* A, uint16_t* A_hi, uint16_t* A_lo, float* A_rs, const float* ln_w, const float* ln_b,
                    int B, int Cin, int T, int H, int W, int p, int pt, int first, float eps,
                    omt_stream_t stream);

/* Inverse Rearrange of to_pixels (omnitokenizer.py:1008 / :1015): P [rows, K] -> video (B,Cin,T,H,W). */
int omt_unpatchify(const float* P, float* video, int B, int Cin, int T, int H, int W, int p, int pt,
                   int first, omt_stream_t stream);

/* Un-patchify fused with the consumers' uint8 conversion: u8 = trunc(clamp(x * mul + add, lo, hi) * post), written
 * channels-LAST (B, T, H, W, Cin).  (mul, add, lo, hi, post) = (1, .5, 0, 1, 255) is vqgan_eval.py:139,147-148
 * `(clamp(x_recons + 0.5, 0, 1) * 255).byte()` and Latte's sample_ddp.py:206; (255, 128, 0, 255, 1) is DiT's
 * sample_ddp.py:163.  Each step rounds in fp32 like the torch expression, so the bytes are identical to it. */
int omt_unpatchify_u8(const float* P, uint8_t* out, int B, int Cin, int T, int H, int W, int p, int pt,
                      int first, float mul, float add, float lo, float hi, float post, omt_stream_t stream);

/* PEG (attention.py:298-338) + residual: y[r,:] = x[r,:] + bias + sum_k w[k,:] * x[nbr[r % rows_per_b, k] , :]
 * nbr: int32 [rows_per_b, 27] canonical neighbour rows inside one batch element, -1 = zero padding
 * (the spatial stencil or the reference's literally-reshaped "scrambled" temporal one, built by the host);
 * w27: weights repacked [27, C]. */
int omt_peg(const float* x, float* y, const float* w27, const float* bias, const int32_t* nbr,
            int B, int rows_per_b, int C, omt_stream_t stream);

/* Same operation as omt_peg, tiled: the stencil is evaluated in volume space (t2,h2,w2) with a
 * shared-memory halo tile and a sliding register window (9 loads per output instead of 27).
 * temporal != 0 selects the reference's literally-reshaped '(b h w) t d' volume (attention.py:313-319),
 * causal != 0 pads t by (2,0) instead of (1,1).  x, y: canonical [B*T*h*w, C]. */
int omt_peg_volume(const float* x, float* y, const float* w27, const float* bias, int B, int T, int h, int w,
                   int C, int temporal, int causal, omt_stream_t stream);

/* In-place rope + l2norm + per-dim scale on q and k (attention.py:417-421, :435-437).
 * q[M, heads*64] (ld ldq), k likewise; cos/sin [N, 32] or NULL (no rope; temporal blocks);
 * the rope position of row r is r % N. */
int omt_qk_prep(float* q, int ldq, float* k, int ldk, const float* q_scale, const float* k_scale,
                const float* rope_cos, const float* rope_sin, int M, int N, int heads,
                omt_stream_t stream);

/* Full (non-causal) attention over n_seq sequences of N contiguous canonical rows, head dim 64:
 * o = softmax(scale * q k^T) v   (attention.py:451, SDPA branch: no additive bias).  N % 64 == 0.
 * All three attention cores: when o_hi != NULL the result is written as fp16 hi / lo operand planes
 * (leading dimension ldo) for the out-projection GEMM instead of fp32 o (o may then be NULL). */
int omt_attn_spatial(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                     float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int n_seq, int N, int heads, float scale,
                     omt_stream_t stream);

/* omt_attn_spatial on the operand planes written by omt_linear_h(OMT_EPI_QKV_PLANES): tcgen05 kind::f16 core, Q / P in
 * tensor memory, K / V tiles straight from TMA (V as an MN-major operand: no transpose), N % 128 == 0.
 * qk_plane_scale = q_plane_scale * k_plane_scale; vinv [heads][n_seq * N]. */
int omt_attn_spatial_h(const uint16_t* q_hi, const uint16_t* q_lo, int ldq, const uint16_t* k_hi, const uint16_t* k_lo, int ldk,
                       const uint16_t* v_hi, const uint16_t* v_lo, int ldv, const float* vinv, float qk_plane_scale,
                       float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int n_seq, int N, int heads, float scale,
                       omt_stream_t stream);

/* 8x8 (ws x ws, ws*ws == 64) window attention with relative position bias (attention.py:254-286):
 * o = softmax(scale * q k^T + bias[head]) v within each window of the (h, w) token grid.
 * bias: [heads, 64, 64] already gathered from the 225-entry table. */
int omt_attn_window(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                    float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, const float* bias, int n_frames, int h, int w, int ws, int heads,
                    float scale, omt_stream_t stream);

/* Temporal attention: for every (b, n) a sequence over t' (rows b*T*N + t*N + n), optional causal
 * mask (attention.py:451 is_causal: key j <= query i); any T >= 1, exact fp32 on CUDA cores.
 * T <= 17: one warp per (b, n, head) holds the whole sequence in registers (one instance per T);
 * T > 17: one warp per (b, n, head) and tile of 32 query frames streams K / V through shared memory in
 * chunks of 16 frames with an online softmax.  Either way a result does not depend on B, N or the grid. */
int omt_attn_temporal(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                      float* o, uint16_t* o_hi, uint16_t* o_lo, int ldo, int B, int T, int N, int heads, float scale, int causal,
                      omt_stream_t stream);

/* pre_vq_conv (omnitokenizer.py:144-154) [+ F.normalize(dim=channels) :251-252]:
 * z[M, cd] = x[M, C] . Wt^T + b, cd in {8, 16}; l2 != 0 divides each row by max(||z||, 1e-12). */
int omt_pre_vq(const float* x, int ldx, const float* Wt, const float* b, float* z, int M, int C, int cd,
               int l2, omt_stream_t stream);

/* Codebook.forward nearest-neighbour search (modules/codebook.py:82-86), cd == 8:
 * d[n,k] = (sum z^2 - 2 z.E_k) + sum E_k^2 in that association, idx = first argmin.
 * e2: [n_codes] precomputed sum E^2; n_codes % 32 == 0.  Also accumulates counts[n_codes] (int32, caller zeroes) --
 * the fixed-size replacement of torch.unique (:65).  One launch, no workspace. */
int omt_vq_search(const float* z, const float* E, const float* e2, int M, int n_codes,
                  int64_t* idx, int32_t* counts, omt_stream_t stream);

/* The whole VQ lookup in ONE launch: pre_vq_conv (omnitokenizer.py:248) + F.normalize (:251-252, l2 != 0) + the search
 * above.  x [M, C] is the encoder output; z [M, 8] receives the (normalised) projection (may be NULL).  A cluster of 8
 * CTAs shares a block of 512 rows: each CTA projects 64 of them, broadcasts z through distributed shared memory and
 * searches all 512 against its eighth of the table; per-row minima meet again in the row's owner CTA. */
int omt_vq_fused(const float* x, int ldx, const float* Wt, const float* b, int C, int l2, float* z,
                 const float* E, const float* e2, int M, int n_codes, int64_t* idx, int32_t* counts,
                 omt_stream_t stream);

/* Decode-side lookup: F.embedding gather (omnitokenizer.py:270) + post_vq_conv Linear(cd, C) (:156-160).
 * If idx != NULL rows come from E[idx[r]]; else from zc[M, cd].  X[M, C] = row . Wt^T + b.
 * When z_st_from != NULL (forward(): straight-through, codebook.py:120) the row is (E[idx]-z)+z and is
 * also written to zq_out[M, cd] (may be NULL). */
int omt_post_vq(const int64_t* idx, const float* E, const float* zc, const float* z_st_from,
                float* zq_out, const float* Wt, const float* b, float* X, int M, int C, int cd,
                omt_stream_t stream);

/* ---- f16x3 path: operands as 16-bit planes ------------------------------------------------------------
 * An fp32 matrix X is carried as hi = fp16(X) (round to nearest, saturating) and lo = fp16((X - hi) * 2^11), two
 * uint16 matrices with a common leading dimension: X ~= hi + lo * 2^-11 to 2^-23 |X| for |X| < 65504.
 * Producers below write the planes directly; weights are split once on the host.
 * ROW-SCALED form: a producer that sees whole rows (LayerNorm, patch gather) multiplies the row by the power of two
 * that puts its largest magnitude in [2^14, 2^15) and stores hi = fp16(x'), lo = fp16(x' - hi) UNSCALED plus the inverse
 * scale per row; the weights carry one such scale per matrix.  The GEMM then needs ONE accumulator instead of two
 * (256-wide tiles AND double buffering).  Both A operands of a dual-A call use the same form. */
typedef struct omt_linear_h_args {
  const uint16_t* a_hi; const uint16_t* a_lo;      /* A planes [M, lda] */
  const float* a_rs; const float* a2_rs;           /* non-NULL: ROW-SCALED planes (below): inverse row scales [rows of A] */
  float w_scale;                                   /* row-scaled form: inverse of the per-matrix scale of the W planes */
  const uint16_t* a2_hi; const uint16_t* a2_lo;    /* optional second A (dual-A form, columns >= n_split), same lda / row map */
  int n_split;                                     /* multiple of 256 */
  int lda, a_seg, a_seg_stride, a_seg_off;         /* lda % 8 == 0; row map as in omt_linear (segments of 64 rows) */
  const uint16_t* w_hi; const uint16_t* w_lo;      /* W planes [N rounded up to 256, K], K % 64 == 0 */
  float* c; int ldc, c_seg, c_seg_stride, c_seg_off;   /* fp32 output (OMT_EPI_NONE / OMT_EPI_QKV); row map segments of 32 rows */
  uint16_t* u_hi; uint16_t* u_lo; int ldu;         /* OMT_EPI_GEGLU: output planes U[M, N/2] */
  int M, N, K;
  const float* bias; const float* residual; int ldr;   /* residual may alias c */
  int epilogue;
  const float* q_scale; const float* k_scale; const float* rope_cos; const float* rope_sin;   /* OMT_EPI_QKV, as omt_linear2 */
  int qk_cols, tokens;
  /* OMT_EPI_QKV_PLANES: output planes u_hi / u_lo [M, N] (ldu): q / k heads multiplied by the static powers of two
   * q_plane_scale / k_plane_scale (|q| <= max|q_scale| after l2norm, so the bound is exact), v heads scaled per
   * (row, head) with the inverse scales written to vinv [N_v / 64][M]; lo planes unscaled. */
  float q_plane_scale, k_plane_scale;
  float* vinv;
  /* statically bounded operands: a_rs_uniform > 0 (with a_rs == NULL) = row-scaled form with ONE inverse scale for all rows;
   * u_scale > 0 (OMT_EPI_GEGLU) = write the U planes in that form, multiplied by u_scale (|U| * u_scale < 65504 is the
   * caller's guarantee: |gelu(g) * a| <= |g| |a| and both are bounded through the LayerNorm in front of the GEMM). */
  float a_rs_uniform, u_scale;
} omt_linear_h_args;

/* Same contract as omt_linear / omt_linear2 (nn.Linear + the fused epilogues) on operand planes. */
int omt_linear_h(const omt_linear_h_args* args, omt_stream_t stream);

/* LayerNorm as omt_layernorm with plane outputs for the GEMM that consumes it:
 * y (fp32, may be NULL), (y_hi, y_lo) planes of the normalised row, and optionally (x_hi, x_lo) planes of the RAW
 * input row -- Attention.forward projects k, v from the un-normalised input (attention.py:407-412).  lds = leading
 * dimension of every plane (lds % 8 == 0).  The row map applies to x / y; planes are written at the LOGICAL row.
 * y_rs / x_rs != NULL: that plane pair is written in the row-scaled form and the inverse row scales go to y_rs / x_rs [M]. */
int omt_layernorm_h(const float* x, int ldx, float* y, int ldy, uint16_t* y_hi, uint16_t* y_lo, float* y_rs,
                    uint16_t* x_hi, uint16_t* x_lo, float* x_rs, int lds, const float* w, const float* b,
                    int M, int C, float eps, int seg, int seg_stride, int seg_off, omt_stream_t stream);

/* Tuning knobs (process-wide): "pdl" = 0 (default; measured 2-4 % slower when on) | 1 programmatic dependent launch;
 * "peg_kernel" = 4 (default: cp.async zero-fill halo gather + packed f32x2 FMAs) | 3 (register-staged gather; also the
 * fallback for T > 64 or w > 254); identical bits;
 * "attn_kernel" = 3 (default: tcgen05 spatial attention core when N % 128 == 0) | 1 (CUDA-core fp32);
 * "f16_bn" = 0 (default: by shape) | 256 (256 x 256 tiles, one TMEM buffer released as soon as the epilogue has drained
 * it into registers) | 128 (256 x 128 tiles, double-buffered accumulators): tile width of omt_linear_h's two-accumulator form;
 * "attn_f16_ctas" = 2 (default: single S / P buffers, 256 TMEM columns, two CTAs per SM) | 1 (double-buffered S / P, one CTA per SM):
 * shape of omt_attn_spatial_h's kernel; identical results. */
int omt_set_option(const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* OMNITOK_B200_H_ */
