/*
 * wsr.h -- C ABI of the B200-native diffusion super-resolution hot path (libwsr.so).
 *
 * The reference (jellikus/Super-Resolution-Enhancement-of-Weather-Data-Using-Diffusion-Models) is pure Python/PyTorch
 * and has NO plugin / FFI / operator ABI of its own (SURVEY.md 8b): its seam is the Python class registry
 * models/diffusion_models/networks.py:116-134.  This header is therefore the boundary a maintainer of the
 * reference would bind with ctypes (see INTEGRATION.md); every entry point names the reference code whose arithmetic
 * it replaces.  All pointers are DEVICE pointers unless stated otherwise, all sizes are explicit, outputs and
 * workspaces are caller-owned, `stream` is a cudaStream_t passed as void*.  No torch types, no hidden allocation,
 * no exceptions.  Every function returns 0 on success and a negative WSR_E_* code on failure;
 * wsr_last_error() returns a thread-local description of the last failure.
 *
 * Activations are NHWC ("pixels x channels") with an explicit channel pitch `ld` (elements between consecutive
 * pixels), so a tensor may be a channel slice of a wider buffer (skip-concat without copies, RRDB dense blocks).
 * Conv weights are packed [tap][Cout][Cin] (tap = ky*KW + kx) in the activation dtype.
 */
#ifndef WSR_H_
#define WSR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WSR_OK 0
#define WSR_E_INVALID (-1)     /* invalid argument                      */
#define WSR_E_UNSUPPORTED (-2) /* shape / dtype not supported by kernel */
#define WSR_E_CUDA (-3)        /* CUDA runtime / driver error           */

#define WSR_F32 0
#define WSR_BF16 1

#define WSR_ACT_NONE 0
#define WSR_ACT_LRELU02 1 /* LeakyReLU(0.2), rrdb_encoder/RRDBNet.py:31,103 */
#define WSR_ACT_RELU 2    /* simple_cnn/Simple_CNN.py:17-19                 */
#define WSR_ACT_SWISH 3   /* nn_modules/functional_layers.py:44-47          */
#define WSR_ACT_MISH 4    /* nn_modules/functional_layers.py:49-52          */

const char* wsr_last_error(void);
int wsr_version(void);
/* 1 when the current device is compute capability 10.x (tcgen05 path usable). */
int wsr_device_is_sm100(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Convolution.  Replaces nn.Conv2d call sites: nn_modules/resnet.py:24,51,78-79; functional_layers.py:64,79;
 * resdiff/unet.py:68; guided_cross_attention.py:20-22; fd_info_spliter.py:35; RRDBNet.py:27-36,93-97;
 * Simple_CNN.py:16-20.
 *
 *   y[n,oh,ow,co] = ( act( sum_{tap,ci} w[tap][co][ci] * X[n, ih, iw, ci]
 *                          + sum_{ci2} w2[co][ci2] * x2[n,oh,ow,ci2]          (optional fused 1x1 "res_conv")
 *                          + bias[co] + rowvec[n*rowvec_ld + co] ) ) * out_scale
 *                   + res[n,oh,ow,co] * res_scale + res2[n,oh,ow,co] * res2_scale
 *
 * X is x, or its nearest-neighbour x2 upsampling when `upsample` != 0 (functional_layers.py:62-67); zero padding
 * (ksize-1)/2; stride 1 or 2.  H, W are the dimensions of x; the output is (H*up/stride, W*up/stride).
 * upsample = 1: w holds the 9 original taps (every output phase evaluates all 9, bit-for-bit the reference's sum).
 * upsample = 2: w holds the PHASE-MERGED taps [4 phases][2x2][w_rows][Cin] made by wsr_pack_upsample_weight: taps that
 *               read the same source pixel are pre-summed, 2.25x fewer MACs (weights are summed in fp32, then rounded).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct {
  const void* x;  int x_dtype;  int N, H, W, Cin;  int x_ld;
  const void* w;                                   /* [ksize*ksize][w_rows][Cin], dtype = x_dtype          */
  int w_rows;                                      /* rows per tap in w / w2 (>= Cout, zero padded); 0 = Cout */
  int ksize, stride, upsample;
  int Cout;
  const void* x2; int Cin2; int x2_ld;             /* optional second K segment (1x1), dtype = x_dtype     */
  const void* w2;                                  /* [Cout][Cin2]                                         */
  const float* bias;                               /* [Cout] or NULL                                       */
  const float* rowvec; int rowvec_ld;              /* [N][rowvec_ld] or NULL (time embedding)              */
  int act;
  float out_scale;
  const void* res;  int res_dtype;  int res_ld;  float res_scale;
  const void* res2; int res2_dtype; int res2_ld; float res2_scale;
  void* y; int y_dtype; int y_ld;
  /* optional fused GroupNorm statistics of the OUTPUT: per-(image, channel) sum and sum of squares of y (taken from the
   * fp32 epilogue values, before the store rounding) are ACCUMULATED into gn_stats[n*gn_stats_ld + 2*co + {0,1}] (doubles; see wsr_gn_stats).  NULL = off. */
  double* gn_stats; int gn_stats_ld;
  /* optional fused GroupNorm (+ Swish) of the INPUT (wsr_conv_tc only, layers for which wsr_conv_tc_can_fuse_gn() is 1):
   * the convolution reads the RAW tensor x and applies a = gn_act(x * scale + shift) on its way into shared memory, with
   * gn_table[n*gn_table_ld + c] = (scale, shift) pairs (2 floats) from wsr_gn_finalize; zero padding applies to a.  The
   * optional second segment x2 stays raw.  Replaces the separate GroupNorm+Swish pass of nn_modules/resnet.py:21-22. */
  const float* gn_table; int gn_table_ld; int gn_act;
  /* optional second packing of a 3x3 weight with Cout <= 64 for the "vertical tap merge" of wsr_conv_tc (rows of >= 128
   * pixels): [kx][3 * 64 rows][Cin], row block b of slice kx = the 64 (zero-padded) output channels of tap (ky = 2 - b, kx),
   * dtype = x_dtype (wsr_pack_conv_weight_vmerge).  NULL = not available. */
  const void* w_vmerge;
} WsrConvDesc;

/* fp32-accumulate SIMT implicit GEMM; any dtype, any channel count.  This is the "fp32 check mode" kernel. */
int wsr_conv_simt(const WsrConvDesc* d, void* stream);
/* tcgen05/TMEM implicit GEMM fed by TMA; bf16 operands, fp32 accumulation.  Requires x_dtype = BF16, Cin % 64 == 0,
 * Cin2 % 64 == 0, Cout % 16 == 0, W a power of two (>= 2), pitches % 8 == 0, 16-byte aligned bases. */
int wsr_conv_tc(const WsrConvDesc* d, void* stream);
int wsr_conv_tc_can_fuse_gn(const WsrConvDesc* d);
/* test introspection: (CTA pairs << 20) | (column-tile width << 8) | K splits chosen by the most recent wsr_conv_tc / wsr_conv_taps_tc call.
 * Classic-mode launches whose 3x3 K loop is long (>= 36 K blocks) and whose 64-column tiles fill at most half of the SMs are split
 * over a 2-CTA cluster (each CTA accumulates half of the K blocks; partial tiles are exchanged through distributed shared memory). */
int wsr_debug_last_tc_config(void);
/* CTA pairs (tcgen05 cta_group::2: two SMs of a TPC share one 256 x 256 tile, each staging half of the weight columns) for the classic-mode
 * 256-column convolution tiles: 0 = never, 1 = launches of more than one wave (default), 2 = every eligible launch (an even number of row
 * tiles).  Returns the previous mode.  wsr_debug_last_tc_config() reports the choice in bit 20. */
int wsr_debug_set_pair(int mode);
/* Programmatic dependent launch for the kernels launched after this call (convolutions, GroupNorm apply, small attention, head): a kernel
 * may start its prologue while its predecessor drains.  Off until wsr_set_pdl(1) (no gain at 64 images per GPU, where the device runs under
 * its power cap); the sampling loop switches it on around the graph capture of small batches.  Returns the previous setting (0 or 1). */
int wsr_set_pdl(int on);

/* ---------------------------------------------------------------------------------------------------------------
 * Tap-table convolution: the same kernels driven by an explicit list of taps instead of (ksize, stride, upsample).
 * It expresses every DATA GRADIENT of the path as a forward convolution on flipped / transposed weights (the backward
 * of nn.Conv2d in `l_pix.backward()`, models/diffusion_models/model.py:67): stride-2 Downsample -> four output-phase
 * launches of a transposed convolution; "nearest x2 + conv3x3" Upsample -> one 4x4 stride-2 convolution.
 *   for g in [0,GH) x [0,GW):   y[n, g*out_mul + out_p, co] = epilogue( sum_t sum_ci w[wtap_t][co][ci] * x[n, in_sub*(g + d_t) + p_t, ci] )
 * x is (N, d->H, d->W, Cin), y is (N, OH, OW, Cout); out-of-range input pixels read as zero.  d->ksize / stride /
 * upsample are ignored; the epilogue fields (bias, rowvec, act, res, res2, gn_stats) keep their meaning.
 * ------------------------------------------------------------------------------------------------------------- */
#define WSR_MAX_TAPS 16
typedef struct {
  int GH, GW;                 /* loop grid per image                                              */
  int in_sub;                 /* 1 or 2: input subsampling factor                                 */
  int out_mul, out_py, out_px;/* output pixel = g * out_mul + out_p                                */
  int OH, OW;                 /* output tensor extent                                             */
  int ntaps;
  int py[WSR_MAX_TAPS], px[WSR_MAX_TAPS];   /* input phase of the tap (0 <= p < in_sub)             */
  int dy[WSR_MAX_TAPS], dx[WSR_MAX_TAPS];   /* input offset of the tap on the subsampled grid        */
  int wtap[WSR_MAX_TAPS];                   /* index of the tap's [w_rows][Cin] matrix inside d->w   */
} WsrTapTable;
int wsr_conv_taps_simt(const WsrConvDesc* d, const WsrTapTable* t, void* stream);
/* tcgen05 version; same operand constraints as wsr_conv_tc; in_sub = 2 needs even H, W. */
int wsr_conv_taps_tc(const WsrConvDesc* d, const WsrTapTable* t, void* stream);

/* Weight (and bias) gradient of a tap-table convolution (backward of nn.Conv2d w.r.t. weight / bias):
 *   dw[wtap_t * dw_stap + co * dw_sco + ci * dw_sci] += sum_{n, g} dy[n, g*out_mul + out_p, co] * X[n, in_sub*(g + d_t) + p_t, ci]
 *   dbias[co] += sum_{n, g} dy[n, g*out_mul + out_p, co]
 * X = x, or x read through a nearest x2 upsampling when up == 2 (pixel u reads x[u / 2]; t describes the taps on the
 * upsampled grid).  The explicit dw strides let the result land directly in the reference's OIHW parameter layout. */
typedef struct {
  const void* x;  int x_dtype;  int N, H, W, Cin;  int x_ld;
  const void* dy; int dy_dtype; int Cout; int dy_ld;           /* (N, t->OH, t->OW, Cout) */
  float* dw; int64_t dw_stap, dw_sco, dw_sci;
  float* dbias;                                                /* or NULL */
  int up;                                                      /* 1 or 2 */
} WsrWgradDesc;
int wsr_conv_wgrad_simt(const WsrWgradDesc* d, const WsrTapTable* t, void* stream);
/* tcgen05 version: the reduction runs over pixels, so both operands are consumed MN-major (channel-contiguous NHWC boxes
 * loaded by TMA; no transposed copies).  Requires bf16 x / dy, pitches % 8, 16-byte aligned bases, a table that loops
 * over the whole output (out_mul 1), loop-grid dimensions that form 64-pixel tiles, and dbias == NULL (use
 * wsr_col_sums).  Partial sums of the K splits are added to dw with fp32 reductions. */
int wsr_conv_wgrad_tc(const WsrWgradDesc* d, const WsrTapTable* t, void* stream);
/* out[c] += sum over pixels of x[p][c] (NHWC, pitch x_ld): bias gradients. */
int wsr_col_sums(const void* x, int x_dtype, int64_t pixels, int C, int x_ld, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched GEMM  D[b][m][n] = alpha * sum_k A[b][m][k] * B[b][n][k] (+ bias[n]) (+ res[b][m][n]),
 * used for the attention products (nn_modules/resnet.py:90-97, guided_cross_attention.py:34-41) and the linear
 * layers.  Element strides are explicit; the tcgen05 version requires unit k-stride for both operands.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct {
  const void* a; int a_dtype; int64_t a_sb, a_sm, a_sk;
  const void* b; int b_dtype; int64_t b_sb, b_sn, b_sk;
  void* d; int d_dtype; int64_t d_sb, d_sm, d_sn;
  const void* res; int res_dtype; int64_t res_sb, res_sm, res_sn;
  const float* bias;
  int batch, M, N, K;
  float alpha;
} WsrGemmDesc;

int wsr_gemm_simt(const WsrGemmDesc* d, void* stream);
int wsr_gemm_tc(const WsrGemmDesc* d, void* stream);

/* Fused single-head attention O = softmax(scale * Q K^T) V on tcgen05/TMEM; the (Nq x Nk) score matrix stays on chip.
 * Replaces nn_modules/resnet.py:90-97 and resdiff/guided_cross_attention.py:34-41 (scale = 1/sqrt(C)).
 * q (B,Nq,d) pitch q_ld; k (B,Nk,d) pitch k_ld; vT (B,d,Nk) = V transposed, dense; o (B,Nq,d) pitch o_ld; all bf16.
 * Requires d in {64,128}, Nq % 128 == 0, Nk % 128 == 0, pitches % 8 == 0, 16-byte aligned bases. */
int wsr_attention_tc(const void* q, int q_ld, const void* k, int k_ld, const void* vT, void* o, int o_ld, int B, int Nq,
                     int Nk, int d, float scale, void* stream);

/* The same product for SHORT key sequences and WIDE heads (the low-resolution levels): SelfAttention at 16x32 / 8x16
 * (nn_modules/resnet.py:81-100: N = 512 / 128, d = 512) and HF_guided_CA levels 2, 3 (resdiff/guided_cross_attention.py:24-44:
 * N = 512, d = 256; N = 128, d = 512).  The whole 128 x Nk score block sits in tensor memory: exact single-pass softmax, P in
 * shared memory, O re-uses the score columns.  Same argument meaning as wsr_attention_tc.
 * Requires Nq % 128 == 0, 64 <= Nk <= 512 with Nk % 64 == 0, 64 <= d <= 512 with d % 64 == 0 (wsr_attention_small_tc_supported). */
int wsr_attention_small_tc(const void* q, int q_ld, const void* k, int k_ld, const void* vT, void* o, int o_ld, int B, int Nq,
                           int Nk, int d, float scale, void* stream);
/* ... with V as it leaves the q | k | v projection convolution: (B, Nk, d) pixels x channels with pitch v_ld (an MN-major tcgen05
 * operand; no V^T GEMM).  Same shape requirements; v_ld % 8 == 0. */
int wsr_attention_small_nhwc_tc(const void* q, int q_ld, const void* k, int k_ld, const void* v, int v_ld, void* o, int o_ld, int B,
                                int Nq, int Nk, int d, float scale, void* stream);
int wsr_attention_small_tc_supported(int Nq, int Nk, int d);

/* ConvTranspose2d(k=8, s=4, p=2) of srdiff/unet.py:43-45,118.  x NHWC (N,H,W,Cin); w packed [ky*8+kx][Cout][Cin];
 * y NHWC (N,4H,4W,Cout). */
int wsr_conv_transpose_k8s4(const void* x, int x_dtype, int N, int H, int W, int Cin, int x_ld, const void* w,
                            const float* bias, int Cout, void* y, int y_dtype, int y_ld, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * GroupNorm (eps, affine) + activation.  Replaces nn.GroupNorm + Swish of nn_modules/resnet.py:21-22,77 and
 * guided_cross_attention.py:19.  Two kernels: per-(image, channel) sums, then normalise (+act).
 * stats: doubles, stats[n*stats_ld + 2*c + {0,1}] = (sum, sum of squares) of channel c of image n (stats_ld >= 2*C, so
 * the statistics of a channel slice can live inside those of a wider concat buffer); wsr_gn_stats ACCUMULATES (zero
 * the buffer first with wsr_fill_zero).  The convolution kernels can produce the same statistics in their epilogue
 * (WsrConvDesc.gn_stats), which removes this read pass.
 * ------------------------------------------------------------------------------------------------------------- */
int wsr_gn_stats(const void* x, int x_dtype, int N, int HW, int C, int x_ld, double* stats, int stats_ld, void* stream);
int wsr_gn_apply(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                 const float* gamma, const float* beta, int groups, float eps, int act, void* y, int y_dtype,
                 int y_ld, void* stream);
/* table[n*table_ld + c] = (gamma_c * rstd, beta_c - mean * gamma_c * rstd) as float pairs (table_ld counts PAIRS), so that
 * GroupNorm(x)*gamma+beta = x*scale+shift; consumed by the fused-input mode of wsr_conv_tc (WsrConvDesc.gn_table). */
int wsr_gn_finalize(const double* stats, int stats_ld, int N, int HW, int C, int groups, float eps, const float* gamma,
                    const float* beta, float* table, int table_ld, void* stream);
int wsr_fill_zero(void* p, int64_t bytes, void* stream);
/* Training-mode Block (nn_modules/resnet.py:21-24: GroupNorm -> Swish -> Dropout -> Conv): wsr_gn_apply followed by
 * dropout, y *= keep / (1 - p); the keep mask is Philox4x32-10(seed, tag) indexed by the logical element (n*HW + pix)*C + c,
 * so the backward pass regenerates it. */
int wsr_gn_apply_dropout(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                         const float* gamma, const float* beta, int groups, float eps, int act, void* y, int y_dtype,
                         int y_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, void* stream);
/* The keep-scale mask (0 or 1/(1-p)) that wsr_gn_apply_dropout / wsr_gn_bwd_* apply for (seed, tag): out is NHWC-dense
 * (N, HW, C) fp32, element ((n*HW + p)*C + c).  Test infrastructure for the dropout-on gradient parity check: the mask is exported
 * to the oracle, which multiplies with it where the reference applies nn.Dropout (nn_modules/resnet.py:23). */
int wsr_dropout_mask(float* out, int N, int HW, int C, float p, uint64_t seed, uint32_t tag, void* stream);
/* Backward of GroupNorm + activation (+ dropout).  da = gradient w.r.t. the block output, same dtype as x.
 *   pass 1: red[n*red_ld + 2c + {0,1}] += (sum_p dz, sum_p dz*xhat), dz = da * drop * act'(z)   (doubles, zeroed by the caller)
 *   pass 2: dx (=, or += when accumulate) rstd * (dz*gamma - A_g/m - xhat*B_g/m); dgamma += sum_n red1, dbeta += sum_n red0
 *           (both or neither NULL); colsum[n*colsum_ld + c] = sum_p dx[n,p,c] of THIS contribution (closed form), or NULL. */
int wsr_gn_bwd_reduce(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                      const float* gamma, const float* beta, int groups, float eps, int act, const void* da, int da_dtype,
                      int da_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, double* red, int red_ld, void* stream);
int wsr_gn_bwd_apply(const void* x, int x_dtype, int N, int HW, int C, int x_ld, const double* stats, int stats_ld,
                     const float* gamma, const float* beta, int groups, float eps, int act, const void* da, int da_dtype,
                     int da_ld, float drop_p, uint64_t drop_seed, uint32_t drop_tag, const double* red, int red_ld, void* dx,
                     int dx_dtype, int dx_ld, int accumulate, float* dgamma, float* dbeta, float* colsum, int colsum_ld,
                     void* stream);

/* Row softmax: p[r][:] = softmax(scale * s[r][:]) over `cols`, rows = batch*Nq (resnet.py:92-95). */
int wsr_softmax_rows(const void* s, int s_dtype, int64_t rows, int cols, int64_t s_ld, float scale, void* p,
                     int p_dtype, int64_t p_ld, void* stream);

/* Softmax backward: ds[r][c] = scale * p[r][c] * (dp[r][c] - sum_c' dp[r][c'] * p[r][c']) (backward of resnet.py:92-95). */
int wsr_softmax_bwd_rows(const void* p, int p_dtype, const void* dp, int dp_dtype, int64_t rows, int cols, int64_t ld,
                         float scale, void* ds, int ds_dtype, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Layout / packing helpers.
 * ------------------------------------------------------------------------------------------------------------- */
/* fp32 NCHW -> NHWC slice (dst pitch ld, already offset to the first channel). */
int wsr_nchw_to_nhwc(const float* src, int N, int C, int H, int W, void* dst, int dst_dtype, int dst_ld, void* stream);
int wsr_nhwc_to_nchw(const void* src, int src_dtype, int src_ld, int N, int C, int H, int W, float* dst, void* stream);
/* OIHW fp32 -> [tap][Cout_pad][Cin_pad] (zero padded). */
int wsr_pack_conv_weight(const float* w_oihw, int Cout, int Cin, int KH, int KW, void* dst, int dst_dtype,
                         int Cout_pad, int Cin_pad, void* stream);
/* OIHW fp32 (Cout <= 64, Cin, 3, 3) -> [kx][3*64][Cin_pad] with row block b = tap (ky = 2 - b, kx), rows >= Cout zero. */
int wsr_pack_conv_weight_vmerge(const float* w_oihw, int Cout, int Cin, void* dst, int dst_dtype, int Cin_pad, void* stream);
/* Phase-merged weights of "nearest x2 upsample + conv3x3": OIHW fp32 (Cout,Cin,3,3) -> [phase*4 + a*2 + b][Cout_pad][Cin_pad],
 * phase = py*2+px; (a, b) index the source offsets {-1,0} (py/px = 0) or {0,+1} (py/px = 1). */
int wsr_pack_upsample_weight(const float* w_oihw, int Cout, int Cin, void* dst, int dst_dtype, int Cout_pad, int Cin_pad,
                             void* stream);
/* ConvTranspose2d weight (Cin, Cout, KH, KW) fp32 -> [tap][Cout][Cin]. */
int wsr_pack_convT_weight(const float* w_iohw, int Cin, int Cout, int KH, int KW, void* dst, int dst_dtype, void* stream);
/* Batched re-pack: ONE launch refreshes every packed weight of a plan from the fp32 parameters (the training loop calls it
 * after each optimizer step instead of ~350 per-tensor pack launches).  `jobs_device` is a device array, sorted by
 * `first_unit` (prefix sum of the jobs' unit counts: Cout_pad*Cin_pad pairs for the weight kinds, Cout elements for COPY).
 * `transposed` selects the data-gradient weight W'[o][i][ky][kx] = W[i][o][KH-1-ky][KW-1-kx] of the same parameter (Cout/Cin
 * are the LOGICAL dims of W').  Kinds: CONV = wsr_pack_conv_weight, VMERGE = wsr_pack_conv_weight_vmerge (Cout_pad = 64),
 * UPSAMPLE = wsr_pack_upsample_weight, UPSAMPLE_DGRAD = the 4x4 stride-2 data-gradient taps of "nearest x2 + conv3x3"
 * (always transposed), COPY = dst[i] = src[i] (+ src2[i]) fp32/bf16 vector. */
enum { WSR_PACK_CONV = 0, WSR_PACK_VMERGE = 1, WSR_PACK_UPSAMPLE = 2, WSR_PACK_UPSAMPLE_DGRAD = 3, WSR_PACK_COPY = 4 };
typedef struct WsrPackJob {
  const float* src;
  const float* src2;
  void* dst;
  int64_t first_unit;
  int32_t kind, transposed, dst_dtype, Cout, Cin, taps, Cout_pad, Cin_pad;
} WsrPackJob;
int wsr_repack_batch(const WsrPackJob* jobs_device, int njobs, int64_t total_units, void* stream);
/* dst[i] = (T) src[i] */
int wsr_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, void* stream);
/* nearest x2 upsample of an NHWC tensor (functional_layers.py:62). */
int wsr_upsample2x(const void* x, int dtype, int N, int H, int W, int C, int x_ld, void* y, int y_ld, void* stream);
/* y[...] = a*x + b*z elementwise on NHWC slices (C channels), used for "x + cond" (srdiff/unet.py:126-127). */
int wsr_axpby(const void* x, int x_dtype, int x_ld, float a, const void* z, int z_dtype, int z_ld, float b, void* y,
              int y_dtype, int y_ld, int64_t pixels, int C, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Noise-level embedding.  Replaces PositionalEncoding + noise_level_mlp (functional_layers.py:33-41,
 * resdiff/unet.py:46-53,135; Mish variant srdiff/unet.py:49-54) and the 27 FeatureWiseAffine linears
 * (nn_modules/resnet.py:145-157) plus fd_spliter.noise_func (fd_info_spliter.py:24,43).
 *   level [R] -> temb [R][inner] -> proj [R][P] = temb @ Wcat^T + bcat       (Wcat: [P][inner], all linears stacked)
 * R is the number of rows: the batch in training, or T (all time steps, precomputed once) in sampling.
 * ------------------------------------------------------------------------------------------------------------- */
int wsr_noise_embed(const float* level, int R, int inner, const float* w1, const float* b1, const float* w2,
                    const float* b2, int act, float* temb, void* stream);
int wsr_linear_rows(const float* x, int R, int K, const float* w, const float* bias, int P, float* y, void* stream);

/* Backward of wsr_noise_embed (all four parameter gradients are ACCUMULATED) and of wsr_linear_rows
 * (dx is written, dw / db are accumulated; any of dx, dw may be NULL). */
int wsr_noise_embed_bwd(const float* level, int R, int inner, const float* w1, const float* b1, const float* w2, int act,
                        const float* dtemb, float* dw1, float* db1, float* dw2, float* db2, void* stream);
int wsr_linear_rows_bwd(const float* x, int R, int K, const float* w, const float* dy, int P, float* dx, float* dw,
                        float* db, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * FD_Info_Spliter (resdiff/fd_info_spliter.py:37-117) and the Haar queries (resdiff/unet.py:124-132).
 * ------------------------------------------------------------------------------------------------------------- */
/* Condition-only branch, hoisted out of the T-step loop.  cond: fp32 NCHW (B,C,H,W).  Reproduces the 4-D fftn over
 * (B,C,H,W), the ResSE-derived sigma, the Gaussian high-pass on the unshifted spectrum, x_lf and x_hf.
 * Outputs lf, hf: fp32 NCHW (B,C,H,W).  work: caller scratch of wsr_fd_precompute_workspace_bytes(). */
int64_t wsr_fd_precompute_workspace_bytes(int B, int C, int H, int W);
int wsr_fd_precompute(const float* cond, int B, int C, int H, int W, const float* sigma_fc0, const float* sigma_fc2,
                      const float* hf_fc0, const float* hf_fc2, const float* ct_w, const float* ct_b, int out_ch,
                      float* lf, float* hf, void* work, void* stream);
/* Per-step gate (fd_info_spliter.py:43-47): ne = noise_func(t_emb) is passed in as ne_rows[r][W] (a slice of the
 * wsr_linear_rows output, pitch ne_ld); gate[b][c][w] = ne[w] * (1 + sigmoid(fc2 relu(fc0 mean_w ne))[c]).
 * row_index: device int* giving the row r of ne_rows to use for every b (sampling: the current step), or NULL for r=b. */
int wsr_fd_gate(const float* ne_rows, int ne_ld, const int* row_index, int B, int C, int W, const float* fc0,
                const float* fc2, int hidden, float* gate, void* stream);
/* Backward of the gate (wsr_fd_gate + stem channel block 2, denoise_x = x * gate).  dxin: gradient of the stem input,
 * NHWC pitch d_ld, channels [ch0, ch0+C) hold d denoise_x; x: fp32 NCHW x_t; ne_rows as in wsr_fd_gate with r = b.
 * Writes dne[b*dne_ld + w] and accumulates dfc0 / dfc2 (noise_resSE.fc.{0,2}.weight). */
int wsr_fd_gate_bwd(const void* dxin, int d_dtype, int d_ld, int ch0, const float* x, const float* ne_rows, int ne_ld, int B,
                    int C, int H, int W, const float* fc0, const float* fc2, int hidden, float* dne, int dne_ld, float* dfc0,
                    float* dfc2, void* stream);
/* Backward of the condition-only branch (wsr_fd_precompute) w.r.t. its 3 parameter groups.  g_lf, g_hf: fp32 NCHW
 * gradients of the lf / hf stem channels; `work` must be the workspace the forward call left behind (it keeps the
 * unfiltered spectrum, sigma, the squeeze-excite vectors and the complex inverse transform); `bwork`: scratch of
 * wsr_fd_backward_workspace_bytes().  All parameter gradients are ACCUMULATED. */
int64_t wsr_fd_backward_workspace_bytes(int B, int C, int H, int W);
int wsr_fd_backward(const float* cond, int B, int C, int H, int W, const float* sigma_fc0, const float* sigma_fc2,
                    const float* hf_fc0, const float* hf_fc2, const float* ct_w, const float* g_lf, const float* g_hf,
                    const void* work, void* bwork, float* d_sigma_fc0, float* d_sigma_fc2, float* d_hf_fc0, float* d_hf_fc2,
                    float* d_ct_w, float* d_ct_b, void* stream);
/* Stem input assembly: writes NHWC channels [x, cond, x*gate, lf, hf] (5*C, fd_info_spliter.py:117), zero-pads up
 * to Cpad channels.  x, cond, lf, hf: fp32 NCHW.  Only the first roundup(5*C, 8) (bf16) / 5*C (fp32) channels are
 * written: the caller zero-fills the pad channels of y once. */
int wsr_stem_assemble(const float* x, const float* cond, const float* gate, const float* lf, const float* hf, int B,
                      int C, int H, int W, void* y, int y_dtype, int Cpad, void* stream);
/* Haar detail-band sums for `levels` levels: out[j] fp32 NCHW (B,C,H>>(j+1),W>>(j+1)) packed back to back in `out`;
 * ll_work: scratch of B*C*H*W/4*... floats (>= B*C*H*W/2 floats). */
int wsr_haar_detail_sums(const float* img, int B, int C, int H, int W, int levels, float* out, float* ll_work, void* stream);
/* PhyDiff variant (phydiff/unet.py:265-276): the three detail bands kept apart, out[j] fp32 NCHW (B, 3*C, H>>(j+1), W>>(j+1)) with
 * channel k*C + c = band k (LH, HL, HH) of image channel c; same packing and scratch as wsr_haar_detail_sums. */
int wsr_haar_detail_bands(const float* img, int B, int C, int H, int W, int levels, float* out, float* ll_work, void* stream);
/* PhyDiff stencil channels (phydiff/unet.py:189-196,311-314): F.conv2d(reflect_pad(cond), k) for k = x forward difference,
 * y forward difference, 5-point Laplacian, each with a (1, C, 3, 3) kernel (sum over channels).  out fp32 NCHW (B, 3, H, W). */
int wsr_phy_stencils(const float* cond, int B, int C, int H, int W, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * The steps either side of the sampling loop (SURVEY.md 8f N2), fp32 NCHW planes (plane = one (sample, variable) image).
 * ------------------------------------------------------------------------------------------------------------- */
/* F.interpolate(x, scale_factor=scale, mode="bicubic") of the collate (data/dataset_builder.py:374-380): A = -0.75,
 * align_corners=False, border taps clamped.  src (planes, h, w) -> dst (planes, h*scale, w*scale). */
int wsr_bicubic_upsample(const float* src, int planes, int h, int w, int scale, float* dst, void* stream);
/* StandardScaling.transform / .revert (data/transforms.py:391-409) with per-plane statistics (the reference picks them per
 * sample by month and per variable, transforms.py:116-138): inverse = 0: (x - mean) / std; inverse = 1: std * x + mean. */
int wsr_standard_scale(const float* x, int planes, int64_t hw, const float* mean, const float* stdv, int inverse, float* y, void* stream);
/* One pass for MAE / MSE / RMSE / MR (training/metrics.py:75-201): acc[0] += sum |d|, acc[1] += sum d^2, acc[2] += sum d (doubles),
 * d = scale[plane] * (pred - target); scale = per-plane std folds the inverse transform in (the means cancel), or NULL. */
int wsr_error_sums(const float* pred, const float* target, int planes, int64_t hw, const float* scale, double* acc, void* stream);
/* Probabilistic scores of an ensemble, one pass.  ens: N members (2 <= N <= 256), member-major, member i's planes at
 * ens + i * member_stride (fp32, planes * hw each: the layout of an N x B reverse-loop batch).  Per pixel, over the members x_i:
 *   mean[p*hw + j] = (1/N) sum_i x_i,  spread[p*hw + j] = sqrt(sum_i (x_i - mean)^2 / (N - 1))      (input units; either may be NULL)
 * and ACCUMULATED per plane p into acc[p*5 + k] (doubles, zeroed by the caller), with s = scale[p] (or 1 when scale is NULL):
 *   k = 0: s * (1/N) sum_i |x_i - y|       k = 1: s * sum_i sum_j |x_i - x_j|  (= 2 sum_k (2k - N + 1) x_(k), x_(k) sorted ascending)
 *   k = 2: s^2 * (mean - y)^2              k = 3: s^2 * sum_i (x_i - mean)^2 / (N - 1)              k = 4: s * (mean - y)
 * so CRPS = acc0/n - acc1/(2 N^2 n) (standard) or acc0/n - acc1/(2 N (N-1) n) (fair) over n pixels.  Without target (NULL) only k = 3
 * is accumulated.  rank_hist (or NULL; needs target): rank_hist[p*(N+1) + r] += 1 for every pixel whose target has r members STRICTLY
 * below it -- members equal to the target count as not below.  scale folds the inverse StandardScaling in, as in wsr_error_sums. */
int wsr_ensemble_stats(const float* ens, int N, int64_t member_stride, const float* target, int planes, int64_t hw, const float* scale,
                       float* mean, float* spread, double* acc, unsigned long long* rank_hist, void* stream);
/* Zonal power spectra and row error sums (training.metrics.FieldScores).  pred, target: fp32 (planes, H, W), W along longitude
 * (periodic).  Physical field x = scale[p] * in + shift[p] (scale NULL: 1, shift NULL: 0), error d = scale[p] * (pred - target).  Per
 * (plane p, row r), with X_k = sum_n x_n exp(-2 pi i k n / W) and c_0 = c_{W/2} = 1, c_k = 2 otherwise, the one-sided power
 * P_k = c_k |X_k|^2 / W^2, k = 0 .. W/2 (so sum_k P_k = mean_n x_n^2), is ADDED (doubles) to acc[(p*H + r)*S + j], S = 3*(W/2+1) + 3:
 *   j = k: P of pred      j = (W/2+1) + k: P of target      j = 2*(W/2+1) + k: P of d      j = 3*(W/2+1) + {0,1,2}: sum |d|, sum d^2, sum d
 * A NULL target touches only the pred slots.  Direct DFT in double; one CTA per (plane, row), no atomics (repeated calls are
 * bit-identical).  Nothing is written, and WSR_E_INVALID / WSR_E_UNSUPPORTED returned, for a NULL pred or acc, planes or H below 1,
 * or W odd, below 4 or above 2048. */
int wsr_zonal_spectra(const float* pred, const float* target, int planes, int H, int W, const float* scale, const float* shift, double* acc,
                      void* stream);

/* Prior pre-training (SURVEY.md 8f N4).  image_compare_loss of models/simple_cnn/loss.py:60-76: alpha * fft_mse_loss +
 * beta * dwt_mse_loss (4 Haar levels) between x and y, fp32 NCHW planes with H, W multiples of 16.  *loss += value (double);
 * grad (optional, same shape as x) = d loss / d x.  No FFT is executed: see csrc/pretrain.cu. */
int wsr_image_compare_loss(const float* x, const float* y, int planes, int H, int W, float alpha, float beta, double* loss,
                           float* grad, void* stream);
/* Backward of nn.ReLU(inplace=True) (models/simple_cnn/Simple_CNN.py:17,19) from the kept OUTPUT y: dy[i] = 0 where y[i] <= 0. */
int wsr_relu_mask(const float* y, float* dy, int64_t n, void* stream);
/* Backward of LeakyReLU(slope) (models/rrdb_encoder/RRDBNet.py:105-110,49-53) from the kept OUTPUT y on NHWC channel slices
 * (rows x C, row pitches y_ld / dy_ld): dy[r][c] *= slope where y[r][c] <= 0. */
int wsr_lrelu_mask(const void* y, int y_dtype, int y_ld, void* dy, int dy_dtype, int dy_ld, int64_t rows, int C, float slope, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * DDPM process kernels (models/diffusion_models/diffusion.py).
 * ------------------------------------------------------------------------------------------------------------- */
/* Fused reverse step (diffusion.py:124-125,139-141,168-169,191-192):
 *   x0 = clamp(c_recip[t]*x - c_recipm1[t]*eps, -1, 1); mean = coef1[t]*x0 + coef2[t]*x;
 *   x_out = mean + (t>0 ? z * exp(0.5*logvar[t]) : 0)
 * tables: float [5][T] = (sqrt_recip, sqrt_recipm1, coef1, coef2, logvar).  t_dev: device int* (current step; the
 * kernel does NOT modify it).  z: injected noise (fp32, same shape) or NULL to draw it in-kernel (Philox4x32-10,
 * key = seed, counter = (t, element)).  With z != NULL the step's noise is read at z + (T - t) * z_step_stride, i.e.
 * z may be the whole injected chain [T+1][n] of the parity tests (stride n) or a single tensor (stride 0).
 * eps may be fp32 or bf16 (NHWC with C==1 equals NCHW).  x_out may alias x. */
int wsr_sampler_step(const float* x, const void* eps, int eps_dtype, const float* z, int64_t z_step_stride,
                     uint64_t seed, const float* tables, int T, const int* t_dev, int clip, float* x_out, int64_t n,
                     void* stream);
/* The UNet head fused with the reverse step (SURVEY 8b `final_conv_sampler_step`): eps_hat = conv3x3(Swish(GroupNorm(x))) --
 * `final_conv` of resdiff/unet.py:119,177 (nn_modules/resnet.py:19-28 Block) -- followed, in the same kernel, by the update of
 * wsr_sampler_step on the fp32 NCHW state.  x: RAW (pre-GroupNorm) NHWC bf16 (B,H,W,Cin) with pitch x_ld; stats: the
 * per-(image, channel) (sum, sumsq) doubles the producing convolution emitted; w: the bf16 blocks made by wsr_pack_head_weight from
 * the fp32 [9][Cout][Cin] packing ((Cin / 64) * 9216 bytes); eps_out (optional): fp32 NCHW
 * (B,Cout,H,W); x_state (optional): fp32 NCHW, updated in place with the same Philox stream layout / injected-noise addressing as
 * wsr_sampler_step.  Requires Cin % 64 == 0, Cout <= 4 (wsr_head_sampler_supported). */
int wsr_final_conv_sampler_step(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats, int stats_ld,
                                const float* gamma, const float* beta, int groups, float gn_eps, const void* w,
                                const float* bias, int Cout, float* eps_out, float* x_state, const float* z,
                                int64_t z_step_stride, uint64_t seed, const float* tables, int T, const int* t_dev, int clip,
                                void* stream);
/* Member-keyed (ensemble) variants of wsr_sampler_step, wsr_final_conv_sampler_step and wsr_randn: the batch is a stack of members of
 * member_elems elements each (C*H*W*B_cond), and element i draws from Philox key member_keys[i / member_elems] (device array) at the
 * member-local element i % member_elems instead of key `seed` at element i.  So the slice of member m is bit-identical to the plain entry
 * point run on that slice alone with seed = member_keys[m], however the members are batched.  member_elems must be a positive multiple
 * of 4 (a Philox group of 4 elements never straddles two members); other values return WSR_E_INVALID.  Injected noise (z) ignores the keys. */
int wsr_sampler_step_members(const float* x, const void* eps, int eps_dtype, const float* z, int64_t z_step_stride,
                             const uint64_t* member_keys, int64_t member_elems, const float* tables, int T, const int* t_dev, int clip,
                             float* x_out, int64_t n, void* stream);
int wsr_final_conv_sampler_step_members(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats, int stats_ld,
                                        const float* gamma, const float* beta, int groups, float gn_eps, const void* w,
                                        const float* bias, int Cout, float* eps_out, float* x_state, const float* z,
                                        int64_t z_step_stride, const uint64_t* member_keys, int64_t member_elems, const float* tables,
                                        int T, const int* t_dev, int clip, void* stream);
/* Multistep (DPM-Solver++(2M)) variants of wsr_sampler_step and wsr_final_conv_sampler_step.  tables: float [5][S] =
 * (c_recip, c_recipm1, c_x0, c_x, c_prev), row = *t_dev:
 *   x0 = clamp(c_recip*x - c_recipm1*eps, -1, 1); x_out = c_x0*x0 + c_x*x + c_prev*x0_hist; x0_hist = x0
 * x0_hist: fp32, same shape as x, the clamped x0 of the previous step; it is NOT read when the row's c_prev == 0 (first and final
 * steps), so it needs no initialisation.  No noise.  A null x0_hist, tables or (fused) x_state returns WSR_E_INVALID. */
int wsr_sampler_step_multistep(const float* x, const void* eps, int eps_dtype, float* x0_hist, const float* tables, int S,
                               const int* t_dev, int clip, float* x_out, int64_t n, void* stream);
int wsr_final_conv_sampler_step_multistep(const void* x, int x_ld, int B, int H, int W, int Cin, const double* stats, int stats_ld,
                                          const float* gamma, const float* beta, int groups, float gn_eps, const void* w,
                                          const float* bias, int Cout, float* eps_out, float* x_state, float* x0_hist,
                                          const float* tables, int S, const int* t_dev, int clip, void* stream);
int wsr_head_sampler_supported(int Cin, int Cout, int groups);
int wsr_pack_head_weight(const float* w_tap_cout_cin, int Cout, int Cin, void* dst, void* stream);
/* out[b][:] = table[r][:] for b < B, r = *row_index (one row of the per-time-step projection table broadcast to the
 * batch; lets a captured CUDA graph follow the device-side step counter). */
int wsr_broadcast_row(const float* table, int P, const int* row_index, int B, float* out, void* stream);
/* *t_dev += delta (single thread) -- keeps the step counter on the device so a CUDA graph can be replayed. */
int wsr_step_counter_add(int* t_dev, int delta, void* stream);
/* Standard normal fill with the same Philox stream layout as wsr_sampler_step (counter word = `tag`). */
int wsr_randn(float* out, int64_t n, uint64_t seed, uint32_t tag, void* stream);
int wsr_randn_members(float* out, int64_t n, const uint64_t* member_keys, int64_t member_elems, uint32_t tag, void* stream);
/* q_sample (diffusion.py:209-228): x_noisy = a[b]*(hr-sr) + sqrt(1-a[b]^2)*noise, per-sample a; fp32 NCHW. */
int wsr_q_sample(const float* hr, const float* sr, const float* noise, const float* a, int B, int64_t per_sample,
                 float* x_noisy, void* stream);
/* Sum-reduced L1 / L2 loss between noise and eps_hat (diffusion.py:105-108): *loss += sum |noise-eps|^p.
 * Also writes dloss/deps * scale into grad (or NULL): -sign(noise-eps)*scale (L1), -2(noise-eps)*scale (L2). */
int wsr_noise_loss(const float* noise, const float* eps, int64_t n, int l2, double* loss, float* grad, float scale,
                   void* stream);

/* Adam update over a flat fp32 buffer (torch.optim.Adam semantics; model.py:43-44 uses lr, betas (0.9, 0.999), eps 1e-8,
 * weight_decay 0); `step` is the 1-based step count used for the bias corrections.  The hyper-parameters are doubles so that
 * 1 - beta is rounded to fp32 exactly as torch does. */
int wsr_adam_step(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                  double weight_decay, int step, void* stream);
/* wsr_adam_step (p, m, v bit-identical) that also updates an exponential moving average of the parameters from the new value
 * p' it has just computed: ema = ema * d + (1 - d) * p', three separately rounded fp32 operations like torch's expression with a
 * Python-float d; d == 0 is an exact copy ema = p' (whatever ema held, NaN included).  The library is built with
 * --use_fast_math, so a denormal result is flushed to zero where torch would keep it.  WSR_E_INVALID, nothing written, for a
 * null pointer, n <= 0, step <= 0, ema_decay outside [0, 1), or an ema range that overlaps p, g, m or v. */
int wsr_adam_step_ema(float* p, const float* g, float* m, float* v, float* ema, int64_t n, double lr, double beta1, double beta2,
                      double eps, double weight_decay, int step, double ema_decay, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WSR_H_ */
