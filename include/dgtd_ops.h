/*
 * dgtd_ops.h -- C ABI of libdgtd_ops.so: hand-written sm_100a kernels for the depth-guided
 * texture-diffusion hot path (reference: twig/model/cod.py:1025-1323, call sites :1467-1505).
 *
 * This is the drop-in boundary.  The reference's operator convention for native code is
 * twig/ops: autograd.Function -> pybind -> CUDA (twig/ops/functions/ms_deform_attn_func.py:19-46,
 * twig/ops/src/vision.cpp:13-16, twig/ops/src/cuda/ms_deform_attn_cuda.cu:20-80).  The hot path
 * itself is pure ATen calls today, so each entry point below names the reference lines it
 * replaces.  INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - plain C types only; every pointer is a DEVICE pointer owned by the caller (PyTorch's
 *    caching allocator); the library allocates nothing and keeps no reference after return;
 *  - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*);
 *    no hidden synchronisation; the current CUDA device is the caller's;
 *  - return value 0 = success, negative = error (message via dgtd_last_error(), thread local);
 *    nothing throws or aborts across the ABI;
 *  - "NHWC" = pixel-major (B,H,W,C) contiguous, "NCHW" = PyTorch default contiguous;
 *  - dtype codes: DGTD_F32 / DGTD_BF16.  fp32 mode is the exact path (CUDA-core FMA,
 *    <=1e-4 of the reference); bf16 mode feeds tcgen05 tensor cores with fp32 accumulation.
 */
#ifndef DGTD_OPS_H_
#define DGTD_OPS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGTD_VERSION 100
#define DGTD_F32 0
#define DGTD_BF16 1

#define DGTD_ACT_NONE 0
#define DGTD_ACT_GELU 1 /* exact erf GELU, cod.py:1098 */
#define DGTD_ACT_RELU 2 /* cod.py:1218 */

typedef void* dgtd_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------------------------- */
int dgtd_version(void);
const char* dgtd_last_error(void);
/* number of kernel launches this library has enqueued since load (bench.py `gpu_launches`) */
int64_t dgtd_launch_count(void);

/* ---- a1: cod.compute_surface_normals, cod.py:96-109 -------------------------------------- */
/* depth (B,1,H,W) -> normals (B,3,H,W), NCHW fp32 */
int dgtd_surface_normals_fwd(const float* depth, float* normals, int B, int H, int W,
                             dgtd_stream_t stream);

/* ---- a2: prompt_encoder.fft, cod.py:1256-1271 -------------------------------------------- */
/* Real part of the low-pass projector for an axis of length n (removed band [-line, line-1]),
 * P (n*n fp32, symmetric circulant), plus sc (2*n fp32): sin and cos of 2*pi*line*a/n, which
 * carry the rank-2 imaginary part.  Built once per image size and cached by the caller. */
int dgtd_lowpass_projector(float* P, float* sc, int n, int line, dgtd_stream_t stream);
/* out = | x - Re(P_h x P_w^T) | per (H,W) plane.  x,out: (planes,H,W) fp32.
 * tmp: planes*H*W floats, coef: planes*4 floats (both scratch). */
int dgtd_fft_highpass_fwd(const float* x, const float* Ph, const float* Pw, const float* sc_h,
                          const float* sc_w, float* tmp, float* coef, float* out, int planes,
                          int H, int W, dgtd_stream_t stream);
/* Same operator with the two projector products on the tcgen05 GEMMs (bf16 mode of the path), fp32-accurate
 * through a two-term bf16 split of both operands (x_hi A_hi + x_hi A_lo + x_lo A_hi).  Each split product is ONE
 * K-concatenated GEMM: [x_hi | x_lo | x_hi] . [A_hi | A_hi | A_lo]^T (one fp32 accumulation in TMEM, no accumulator
 * round trips through HBM).  Ph_cat / Pw_cat: [P_hi | P_hi | P_lo]
 * per row (H x 3H, W x 3W bf16); ws_a: planes*H*W*3 bf16; ws_f32: planes*H*W fp32.  H, W multiples of 8. */
int dgtd_fft_highpass_tc3_fwd(const float* x, const void* Ph_cat, const void* Pw_cat, const float* sc_h, const float* sc_w,
                              void* ws_a, float* ws_f32, float* coef, float* out, int planes, int H, int W,
                              dgtd_stream_t stream);

/* ---- a3..a6 fused: cod.py:1295-1298 + MessagePassing.forward :1189-1206 ------------------- */
/* nearest GxG sample of emb1 -> regressor 1x1 conv (3 -> C*49) + sigmoid -> random-walk
 * normalisation; depth -> (encoder1 1x1 conv o bilinear down) -> C x G x G state; T stencil
 * iterations on chip; 1x1 conv C -> 3.  out_grid: (B,3,G,G).  Optional saves for backward:
 * save_states (B,T+1,C,G,G) and save_wn (B,C,49,G*G).  k is fixed at 7 (cod.py:1181). */
int dgtd_diffusion_front_fwd(const float* emb1, const float* depth, const float* reg_w,
                             const float* reg_b, const float* enc_w, const float* enc_b,
                             const float* conv_w, const float* conv_b, float* out_grid,
                             float* save_states, float* save_wn, int B, int H, int W, int G, int C,
                             int T, dgtd_stream_t stream);

/* ---- a6: MessagePassing core as a stand-alone operator, cod.py:1190-1205 ------------------ */
/* x,out (n,c,h,w), weight (n,wc*49,h,w), wc in {1,c}, NCHW fp32; whole plane kept on chip
 * for all T iterations (h*w <= 1024).  save_states nullable: (n,T+1,c,h,w). */
int dgtd_message_passing_fwd(const float* x, const float* weight, float* out, float* save_states,
                             int n, int c, int h, int w, int wc, int T, float eps,
                             dgtd_stream_t stream);
/* Halo-tiled variant for large maps (the 1024^2 x 256 microbench): x,out NHWC (n,h,w,c),
 * dtype fp32 or bf16 storage (fp32 accumulate); weight (n,49,h,w) fp32 shared by all channels
 * (wc == 1).  One launch per iteration; `tmp` (same size as x) is the ping-pong buffer when
 * T > 1.  c must be a multiple of 64 (fp32) / 128 (bf16). */
int dgtd_message_passing_tiled_fwd(const void* x, const float* weight, void* out, void* tmp,
                                   int n, int h, int w, int c, int T, float eps, int dtype,
                                   dgtd_stream_t stream);
/* The same operator forced onto the CUDA-core (SIMT) kernel, whatever the shape (A/B reference for the tensor path). */
int dgtd_message_passing_tiled_simt_fwd(const void* x, const float* weight, void* out, void* tmp,
                                        int n, int h, int w, int c, int T, float eps, int dtype,
                                        dgtd_stream_t stream);
/* The same operator (cod.py:1201-1205, shared weights) on the TENSOR pipe: per 8x16-pixel tile the step is the
 * banded GEMM Y[128 px, c] = A[128, 336 halo px] . X[336, c] on tcgen05.mma; A holds the 49 normalised weights of
 * each pixel in bf16, X is the NHWC map read through TMA as an MN-major operand.  bf16 storage, c a multiple
 * of 256.  dgtd_message_passing_tiled_fwd dispatches here when the shape qualifies. */
int dgtd_message_passing_tc_fwd(const void* x, const float* weight, void* out, void* tmp,
                                int n, int h, int w, int c, int T, float eps, int dtype,
                                dgtd_stream_t stream);
/* Same operator with the MODEL's per-channel weights generated on chip (SURVEY.md 8d config 4, mode W2):
 * W[c,k,p] = sigmoid(Wr[c*49+k,:] . guide[:,p] + br[c*49+k]) (ShapePropWeightRegressor, cod.py:1051-1060,
 * 1296), normalised over the 49 taps (+eps, cod.py:1201) and applied as the 7x7 zero-padded stencil.
 * x,out NHWC (n,h,w,c) fp32 | bf16 storage; guide (n,3,h,w) fp32 NCHW; packed = dgtd_pack_regressor(Wr, br)
 * (c*49 float4).  fast_sigmoid != 0 uses tanh.approx (|err| <= 2.5e-4).  c multiple of 32. */
int dgtd_pack_regressor(const float* wr, const float* br, float* packed, int c, dgtd_stream_t stream);
int dgtd_message_passing_regress_fwd(const void* x, const float* guide, const float* packed, void* out, void* tmp,
                                     int n, int h, int w, int c, int T, float eps, int dtype, int fast_sigmoid,
                                     dgtd_stream_t stream);
/* backward of the stand-alone operator: grad_out (n,c,h,w) -> grad_x (n,c,h,w) and
 * grad_weight (n,wc*49,h,w) (through the normalisation), from the saved states. */
int dgtd_message_passing_bwd(const float* grad_out, const float* weight, const float* states,
                             float* grad_x, float* grad_weight, int n, int c, int h, int w, int wc,
                             int T, float eps, dgtd_stream_t stream);

/* ---- small NCHW helpers so every nn.Module of the path is callable on its own ------------- */
/* 1x1 conv (+ optional sigmoid) in NCHW: ShapePropWeightRegressor (cod.py:1056-1060),
 * encoder1 (:1249), message_passing.conv (:1188). */
int dgtd_conv1x1_nchw_fwd(const float* x, const float* w, const float* b, float* out, int B,
                          int Cin, int Cout, int HW, int sigmoid, dgtd_stream_t stream);
/* backward of the 1x1 conv: y_out non-NULL = the forward applied the sigmoid (its output is passed
 * back); grad_x / grad_w (+grad_b) are optional outputs.  Deterministic reductions. */
int dgtd_conv1x1_nchw_bwd(const float* grad_out, const float* y_out, const float* x, const float* w,
                          float* grad_x, float* grad_w, float* grad_b, int B, int Cin, int Cout, int HW,
                          dgtd_stream_t stream);
/* adjoint of the bilinear resize (h,w) -> (oh,ow): grad_out (planes,oh,ow) -> grad_x (planes,h,w) */
int dgtd_resize_bilinear_nchw_bwd(const float* grad_out, float* grad_x, int planes, int h, int w, int oh,
                                  int ow, dgtd_stream_t stream);
/* F.interpolate(mode='bilinear', align_corners=False) on NCHW fp32 (cod.py:1207,1298) and
 * nearest (cod.py:1295). */
int dgtd_resize_nchw_fwd(const float* x, float* out, int planes, int h, int w, int oh, int ow,
                         int bilinear, dgtd_stream_t stream);
/* predict head for ground truths of different sizes: x (B,1,h,w) logits -> out (B,1,Hmax,Wmax), where image b is
 * sigmoid(bilinear resize of plane b to sizes[b] = (H_b, W_b)) in the top-left H_b x W_b and 0 elsewhere; bit for bit
 * dgtd_resize_nchw_fwd to (H_b, W_b) then dgtd_sigmoid_fwd (a plane already at (H_b, W_b) is copied).  sizes: device
 * int32 (B, 2), 2 <= H_b <= Hmax and 2 <= W_b <= Wmax; an image whose size breaks that is all NaN. */
int dgtd_resize_sigmoid_sized_fwd(const float* x, float* out, const int32_t* sizes, int B, int h, int w, int Hmax,
                                  int Wmax, dgtd_stream_t stream);
/* custom LayerNorm, cod.py:1041-1049: x viewed as (outer, C, inner); channels_last: inner=1 */
int dgtd_layer_norm_fwd(const float* x, const float* w, const float* b, float* out, int64_t outer,
                        int C, int64_t inner, float eps, dgtd_stream_t stream);

/* ---- a7: `embedding2 + image` (cod.py:1302) + ConvNeXt stem / downsample (:1126-1136) ------ */
/* bilinear up-sample of grid (B,3,G,G) to (H,W) + image (B,3,H,W NCHW) -> conv 4x4/4 ->
 * LayerNorm(channels_first) -> out NHWC (B,H/4,W/4,Cout) fp32.  grid may be NULL. */
int dgtd_stem_fwd(const float* image, const float* grid, int G, const float* w, const float* b,
                  const float* ln_w, const float* ln_b, float* out, int B, int H, int W, int Cout,
                  float eps, dgtd_stream_t stream);
/* per-pixel LayerNorm then 2x2/2 patch gather: x NHWC (B,h,w,C) fp32 -> rows (B*(h/2)*(w/2))
 * of 4C values ordered (dy,dx,c); the following linear with the repacked conv weight is the
 * 2x2 stride-2 conv of cod.py:1134. */
int dgtd_ln_patchify_fwd(const float* x, const float* ln_w, const float* ln_b, void* out,
                         int out_dtype, int B, int h, int w, int C, float eps,
                         dgtd_stream_t stream);

/* ---- a8: convnext_Block, cod.py:1104-1117 ------------------------------------------------- */
/* depthwise 7x7 (pad 3) + channels-last LayerNorm: x NHWC fp32 -> out NHWC (fp32|bf16) */
int dgtd_dwconv7_ln_fwd(const float* x, const float* dw_w, const float* dw_b, const float* ln_w,
                        const float* ln_b, void* out, int out_dtype, int B, int h, int w, int C,
                        float eps, dgtd_stream_t stream);
/* Same operator, large-batch variant: TMA-staged halo tiles (4-D box loads, zero fill = padding)
 * + a row LayerNorm pass.  dw_wT = taps transposed to (49, C); ws = B*h*w*C fp32 scratch for the
 * pre-norm conv output.  C must be a multiple of 128. */
int dgtd_dwconv7_ln_tma_fwd(const float* x, const float* dw_wT, const float* dw_b, const float* ln_w,
                            const float* ln_b, float* ws, void* out, int out_dtype, int B, int h, int w,
                            int C, float eps, dgtd_stream_t stream);
/* bf16-mode front of a block with the LayerNorm FOLDED into pwconv1 (cod.py:1106-1109): y = depthwise 7x7 of x,
 * stored once as bf16 (B,h,w,C) -- no fp32 scratch, no normalised copy -- and stats[pixel] = (mean, rstd) over C of
 * the stored values (eps inside the sqrt).  C multiple of 128. */
int dgtd_dwconv7_stats_tma_fwd(const float* x, const float* dw_wT, const float* dw_b, void* y, float* stats, int B,
                               int h, int w, int C, float eps, dgtd_stream_t stream);
/* GEMM with the row LayerNorm fused in its epilogue (the stem of cod.py:1127-1128 in bf16 mode: conv 4x4/4 as a K = 48
 * GEMM + LayerNorm(channels_first) over the 128 output channels): out (M,128) fp32 = LN(a (M,K) bf16 . w (128,K)^T bf16
 * + bias) * ln_w + ln_b.  N == 128, M >= 256, K % 8 == 0. */
int dgtd_linear_ln_fwd(const void* a, const void* w, const float* bias, const float* ln_w, const float* ln_b, float eps,
                       float* out, int M, int N, int K, dgtd_stream_t stream);
/* Thin projection of an fp32 activation on the tensor pipe without a bf16 copy (the head projections of cod.py:1174,
 * N = 24): out (M,ldo) fp32 = a (M,K) fp32 . w (N,K)^T fp32 + bias, products in TF32 (tcgen05 kind::tf32), fp32
 * accumulation.  N <= 64, N % 8 == 0, K % 4 == 0. */
int dgtd_linear_tf32_fwd(const float* a, const float* w, const float* bias, float* out, int M, int N, int K, int ldo,
                         dgtd_stream_t stream);
/* out[M,N] = act(rstd_m * (a[M,K] . w[N,K]^T - mean_m * col_s[N]) + bias[N]) on tcgen05, a / w bf16:
 * == act(LN(a) . W1^T + b1) when w = W1 * ln_weight (rounded to bf16), col_s[n] = sum_k w[n,k] (of the rounded values),
 * bias = W1 . ln_bias + b1, row_stats[m] = (mean, rstd) of row m of a (float2).  pwconv1 with its LayerNorm folded
 * in (cod.py:1108-1110): the normalised activation never exists in memory. */
int dgtd_linear_lnfold_fwd(const void* a, const void* w, const float* bias, const float* col_s, const float* row_stats,
                           void* out, int M, int N, int K, int ldo, int dtype_out, int act, dgtd_stream_t stream);
/* out = residual + gamma * (GELU(LN(y) . W1^T + b1) . W2^T + b2) in ONE kernel, the (M, 4C) hidden tensor staying in
 * shared memory / TMEM: pwconv1 -> act -> pwconv2 -> layer scale -> residual of convnext_Block (cod.py:1108-1116) in bf16
 * inference mode, LayerNorm folded as in dgtd_linear_lnfold_fwd (w1 = W1 * ln_weight in bf16 (4C, C), col_s, cbias (4C),
 * row_stats (M, 2) from dgtd_dwconv7_stats_tma_fwd); w2 bf16 (C, 4C); residual / out fp32 (M, C), out may alias residual.
 * Built for C = 128 (stage 0) and M a multiple of 128; any other shape returns an error (callers use the two GEMMs). */
int dgtd_convnext_mlp_fused_fwd(const void* y, const float* row_stats, const void* w1, const float* col_s,
                                const float* cbias, const void* w2, const float* b2, const float* gamma,
                                const float* residual, float* out, int64_t M, int C, dgtd_stream_t stream);
/* out[M,N] = act(a[M,K] . w[N,K]^T + bias): pwconv1+GELU (:1109-1110), downsample conv
 * (:1134), head 1x1 convs (:1160,1174).  a/w dtype = dtype_in (fp32: CUDA-core exact path,
 * bf16: tcgen05), out dtype = dtype_out, ldo = row stride of out in elements. */
int dgtd_linear_fwd(const void* a, const void* w, const float* bias, void* out, int M, int N,
                    int K, int ldo, int dtype_in, int dtype_out, int act, dgtd_stream_t stream);
/* out = residual + keep[m / rows_per_sample] * gamma * (a . w^T + bias)   (cod.py:1111-1116;
 * keep = DropPath mask/keep_prob per sample, NULL in eval); residual/out fp32 [M,N]. */
int dgtd_linear_residual_fwd(const void* a, const void* w, const float* bias, const float* gamma,
                             const float* keep, int rows_per_sample, const float* residual,
                             float* out, int M, int N, int K, int dtype_in, dgtd_stream_t stream);

/* ---- a9: ShapePropEncoder head, cod.py:1171-1176 ------------------------------------------ */
/* Per-level 1x1 projections, bilinear up to (h0,w0), concat and 1x1 fusion conv, with the fusion conv folded into
 * the four head projections (a 1x1 conv commutes with the bilinear up-sample):
 * z_i (B*h_i*w_i, C) fp32 = x_i (Wf_i Wh_i)^T + Wf_i bh_i;  out = bias + sum_i up(z_i).  hw = {h0,w0,...,h3,w3}.
 * Writes any of: out_nhwc (B,h0,w0,C) fp32, out_nchw (B,C,h0,w0) fp32, out_pad (B,h0,w0,Cpad) bf16 zero padded
 * to Cpad channels (operand of the tensor-core decoders).  C and Cpad multiples of 4. */
int dgtd_fusion_sum_fwd(const float* z0, const float* z1, const float* z2, const float* z3, const int* hw,
                        const float* bias, float* out_nhwc, float* out_nchw, void* out_pad, int Cpad, int B, int C,
                        dgtd_stream_t stream);

/* ---- a10/a11: ShapePropDecoder convs (cod.py:1216-1222) + prompt injection (:1471) -------- */
/* KxK conv as implicit GEMM on NHWC: x (B,h,w,ldx) -> out (B,oh,ow,ldo);
 * input pixel = o*stride + off + tap, zero outside; w packed (Cout, ks*ks*Cin) tap-major;
 * ks=3,stride=1,off=-1 is the reference conv; ks=4,stride s,off o is the last conv folded
 * with the bilinear down-sample to the PVT token grid (exact, SURVEY.md appendix A), whose
 * NHWC output *is* the (B, H_s*W_s, E_s) token layout of cod.py:1471. */
int dgtd_conv_nhwc_fwd(const void* x, const void* w, const float* bias, void* out, int B, int h,
                       int wd, int Cin, int ldx, int oh, int ow, int Cout, int ldo, int ks,
                       int stride, int off, int act, int dtype_in, int dtype_out,
                       dgtd_stream_t stream);
/* Grouped form (the 16 decoders of the path in one launch): group g reads input channels
 * [g*x_group_stride, +Cin) of x, weight rows [g*w_group_rows, +Cout), bias + g*w_group_rows and
 * writes out + g*out_group_stride (elements).  bf16 (tcgen05) needs Cin == 32 (zero-padded
 * latent channels) and tap-major weights (Cout rows, ks*ks*32).
 * Group-major operands (bf16): x_group_stride == 32 means the groups' 32-channel slices interleave in
 * every pixel row of x (pitch ldx); any larger multiple of 8 means group g is its own dense tensor
 * (B,h,w,ldx) at x + g*x_group_stride.  With groups == 1, out_group_stride > 0 and a pixel pitch ldo < Cout
 * (3x3 stride-1 conv, bf16 output, Cout % 32 == 0) the 32-channel chunk c of the output is written to the dense tensor
 * (B,oh,ow,ldo) at out + c*out_group_stride -- the layout the next grouped conv reads as group-major. */
int dgtd_conv_nhwc_grouped_fwd(const void* x, const void* w, const float* bias, void* out, int B,
                               int h, int wd, int Cin, int ldx, int oh, int ow, int Cout, int ldo,
                               int ks, int stride, int off, int act, int dtype_in, int dtype_out,
                               int groups, int64_t x_group_stride, int w_group_rows,
                               int64_t out_group_stride, dgtd_stream_t stream);
/* generic bilinear resize NHWC (B,h,w,C) -> (B,oh,ow,C) == tokens (B,oh*ow,C) */
int dgtd_resize_nhwc_fwd(const void* x, void* out, int B, int h, int w, int C, int oh, int ow,
                         int dtype_in, int dtype_out, dgtd_stream_t stream);

/* ---- training path (config/sod.yml): backward of the trunk / decoders, exact fp32 --------------
 * Gradient GEMMs reuse the CUDA-core GEMM with transposed operand loaders; every reduction is
 * fixed-order (bit-stable gradients).  keep/gamma (nullable) fold the DropPath and layer-scale
 * factors of cod.py:1112-1116 into the operand load. */
/* dx[M,K] (+)= (keep.gamma.g)[M,N] . W[N,K]   (. gelu'(pre[M,K]) when pre != NULL) */
int dgtd_linear_dgrad(const float* g, const float* w, float* dx, const float* pre, const float* keep,
                      const float* gamma, int rows_per_sample, int M, int N, int K, int accumulate,
                      dgtd_stream_t stream);
/* dw[N,K] = (keep.g)^T . a   (split over rows + reduce; ws: dgtd_linear_wgrad_ws_floats floats).
 * ks > 0: `a` is an NHWC tensor read through the im2col view of dgtd_conv_nhwc_fwd (conv wgrad). */
int dgtd_linear_wgrad(const float* g, const float* a, float* dw, float* ws, const float* keep, int rows_per_sample,
                      int M, int N, int K, int ks, int h, int wd, int Cin, int ldx, int oh, int ow, int stride,
                      int off, dgtd_stream_t stream);
int dgtd_linear_wgrad_ws_floats(int M, int N, int K);
/* out[N] = sum_m keep[m/rows] x[m,n]   (ws: cdiv(M,1024)*N floats) */
int dgtd_colsum(const float* x, const float* keep, int rows_per_sample, float* ws, float* out, int M, int N,
                dgtd_stream_t stream);
/* dW2 = gamma.G, db2 = gamma.s, dgamma_n = sum_k W2_nk G_nk + b2_n s_n  (G = (keep.g)^T.h, s = colsum) */
int dgtd_layer_scale_finalize(const float* G, const float* s, const float* W2, const float* b2, const float* gamma,
                              float* dW2, float* db2, float* dgamma, int N, int K, dgtd_stream_t stream);
int dgtd_gelu_fwd(const float* x, float* out, int64_t n, dgtd_stream_t stream);
int dgtd_relu_bwd(const float* g, const float* out, float* dx, int64_t n, dgtd_stream_t stream);
/* LayerNorm over rows of C (cod.py:1042-1049) backward: y = pre-norm input, g = dL/d(out) */
int dgtd_ln_rows_bwd(const float* g, const float* y, const float* w, float* dy, float* ws, float* dw, float* db,
                     int64_t rows, int C, float eps, dgtd_stream_t stream);
int dgtd_ln_rows_bwd_ws_floats(int64_t rows, int C);
/* depthwise 7x7 without the LayerNorm: y = conv(x; wT (49,C), bias) (+ add); flip = rotated taps (dgrad) */
int dgtd_dwconv7_fwd(const float* x, const float* wT, const float* bias, const float* add, float* y, int B, int h,
                     int w, int C, int flip, dgtd_stream_t stream);
/* dwT (49,C), db (C) from x and dy;  ws: (B*cdiv(h,8) + 1) * 50 * C floats */
int dgtd_dwconv7_wgrad(const float* x, const float* dy, float* ws, float* dwT, float* db, int B, int h, int w, int C,
                       dgtd_stream_t stream);
/* stem input gather: patches[(b,oy,ox)][ci*16+ky*4+kx] = image + up(grid); and its adjoint */
int dgtd_stem_patchify(const float* image, const float* grid, int G, void* patches, int out_dtype, int B, int H,
                       int W, dgtd_stream_t stream);
int dgtd_stem_unpatchify(const float* dpatches, float* dimg, int B, int H, int W, dgtd_stream_t stream);
/* 2x2/2 patch gather of an NHWC tensor (rows of 4C, order (dy,dx,c)) and its adjoint */
int dgtd_patchify2(const float* x, float* out, int B, int h, int w, int C, dgtd_stream_t stream);
int dgtd_unpatchify2(const float* dp, float* dx, int B, int h, int w, int C, dgtd_stream_t stream);
/* adjoint of dgtd_resize_nhwc_fwd (fp32): g (B,oh,ow,C) -> dx (B,h,w,C) */
int dgtd_resize_nhwc_bwd(const float* g, float* dx, int B, int h, int w, int C, int oh, int ow, int accumulate,
                         dgtd_stream_t stream);

/* ---- bf16 / tensor-core training path of the trunk ------------------------------------------------
 * One-pass operand preparation for the tcgen05 gradient GEMMs.  mode 0: src fp32, v = keep*src
 * (dst also *gamma); mode 1: src bf16, v = gelu(src); mode 2: src = dH bf16, aux = pre-activation
 * bf16, v = src*gelu'(aux).  dst (M x N) and/or dstT (N x M) in bf16. */
int dgtd_transpose_op(const void* src, const void* aux, void* dst, void* dstT, const float* keep, const float* gamma,
                      int rows_per_sample, int M, int N, int mode, dgtd_stream_t stream);
int dgtd_colsum_bf16(const void* x, float* ws, float* out, int M, int N, dgtd_stream_t stream);
/* The element-wise pass of modes 0 / 2 above fused with the column sums of its result (taken before the bf16
 * rounding): dst (M x N bf16) = v, colsum[n] = sum_m v[m,n] -- the bias gradient of pwconv1 (mode 2) and the
 * layer-scale / pwconv2 bias sum (mode 0) without a second pass over the matrix.  Fixed-order (deterministic).
 * ws: dgtd_eltwise_colsum_ws_floats(M, N) floats. */
int dgtd_eltwise_colsum_ws_floats(int M, int N);
int dgtd_eltwise_colsum(const void* src, const void* aux, void* dst, const float* keep, int rows_per_sample, float* ws,
                        float* colsum, int M, int N, int mode, dgtd_stream_t stream);
/* Weight gradient on tcgen05: out (Mo x No fp32, or its transpose) = a[Kr,Mo]^T . b[Kr,No], a / b row-major bf16
 * activation matrices (pitches lda / ldb in elements; column slices allowed), consumed as MN-major tcgen05
 * operands -- dW = dY^T X straight from dY and X.  Split-K over the long row axis Kr + fixed-order reduction.
 * ws: dgtd_wgrad_tc_ws_floats(Mo, No, Kr) floats. */
int dgtd_wgrad_tc_ws_floats(int Mo, int No, int Kr);
int dgtd_wgrad_tc_mn(const void* a, int lda, const void* b, int ldb, float* out, float* ws, int Mo, int No, int Kr,
                     int transpose_out, dgtd_stream_t stream);
/* Decoder-bank backward, data-movement halves (ShapePropDecoder cod.py:1210-1226 + folded injection :1471).
 * col2im: out[b,iy,ix,c] (pixel pitch ldo) = mask > 0 ? sum over the conv taps that read input pixel
 * (iy,ix) of dcol[(b,oy,ox)][(ty*ks+tx)*Ct + c] : 0; mask (nullable, dtype of out, pitch ldm) is the
 * forward ReLU output.  ks = 1 is a strided masked copy.  dtypes DGTD_F32 | DGTD_BF16. */
int dgtd_col2im_nhwc(const void* dcol, int dcol_dtype, int ldc, int Ct, const void* mask, int ldm, void* out,
                     int out_dtype, int ldo, int B, int h, int w, int C, int ks, int stride, int off, int oh, int ow,
                     dgtd_stream_t stream);
/* col[m][tap*C + c] = x[b, oy*stride+off+ty, ox*stride+off+tx, c] (bf16, C-channel slice at x, pixel pitch
 * ldx, zero outside the map), m = (b*oh+oy)*ow+ox: row-major im2col -- an operand of dgtd_wgrad_tc_mn
 * (decoder gradients, C = 32) or the A operand of a patch-embed GEMM (OverlapPatchEmbed, cod.py:976). */
int dgtd_im2col_nhwc(const void* x, int ldx, void* col, int B, int h, int w, int C, int ks, int stride, int off, int oh,
                     int ow, dgtd_stream_t stream);
/* out[m][c] (fp32) = sum_g x[m][g*group_stride + c], c < C */
int dgtd_group_sum(const void* x, int dtype, float* out, int64_t M, int groups, int group_stride, int C,
                   dgtd_stream_t stream);
/* LayerNorm over rows of C (fp32 in, fp32|bf16 out), C a multiple of 128 */
int dgtd_ln_rows_fwd(const float* y, const float* ln_w, const float* ln_b, void* out, int out_dtype, int64_t rows,
                     int C, float eps, dgtd_stream_t stream);

/* ---- dtype / layout plumbing -------------------------------------------------------------- */
int dgtd_cast_fwd(const void* src, void* dst, int64_t n, int dtype_src, int dtype_dst,
                  dgtd_stream_t stream);
/* NHWC (B,h,w,ldx>=C) any dtype -> NCHW (B,C,h,w) fp32 */
int dgtd_nhwc_to_nchw_fwd(const void* x, float* out, int B, int h, int w, int C, int ldx,
                          int dtype_in, dgtd_stream_t stream);
int dgtd_nchw_to_nhwc_fwd(const float* x, void* out, int B, int h, int w, int C, int ldo,
                          int dtype_out, dgtd_stream_t stream);

/* ---- PVT-v2 blocks consuming the prompts (SURVEY.md 8f-1; cod.py:824-961, 1455-1509): non-GEMM pieces ----
 * ln_tokens: out = LayerNorm_C(x + add) * ln_w + ln_b per token row; sum_out (nullable fp32) = x + add
 * (`x + prompt[i]`, cod.py:1472, fused with norm1 :958).  add nullable, fp32 | bf16; out fp32 | bf16. */
int dgtd_ln_tokens_fwd(const float* x, const void* add, int add_dtype, float* sum_out, const float* ln_w,
                       const float* ln_b, void* out, int out_dtype, int64_t rows, int C, float eps,
                       dgtd_stream_t stream);
/* spatial-reduction conv (k = stride = sr, cod.py:887,903) as a gather: out[(b,oy,ox)][(ty*sr+tx)*C + c] */
int dgtd_patchify_tokens_fwd(const void* x, void* out, int dtype, int B, int h, int w, int C, int sr,
                             dgtd_stream_t stream);
/* Mlp.dwconv + act (cod.py:852-854): depthwise 3x3 pad 1 + bias + GELU(erf) on (B,h,w,C) tokens; wT (9,C) */
int dgtd_dwconv3_gelu_fwd(const void* x, const float* wT, const float* bias, void* out, int dtype, int B, int h, int w,
                          int C, dgtd_stream_t stream);
/* The depthwise 3x3 without the activation: DWConv.forward (cod.py:1520-1531) called on its own. */
int dgtd_dwconv3_fwd(const void* x, const float* wT, const float* bias, void* out, int dtype, int B, int h, int w, int C,
                     dgtd_stream_t stream);
/* Attention core (cod.py:911-915), head_dim 64: q (B*N, heads*64), kv (B*Nk, 2*heads*64) [k | v], out like q;
 * softmax(scale * q k^T) v in fp32 with an online softmax over key tiles. */
int dgtd_attention_fwd(const void* q, const void* kv, void* out, int dtype, int B, int N, int Nk, int heads,
                       float scale, dgtd_stream_t stream);
/* Backward of the attention core (training of the PVT blocks, cod.py:911-915 under autograd): q / kv / out as in
 * dgtd_attention_fwd (dtype fp32 | bf16), dout (B*N, heads*64) fp32 -> dq (B*N, heads*64) and dkv (B*Nk, 2*heads*64)
 * [dk | dv], both fp32.  bf16 inputs: warp-level tensor-core kernels (csrc/attn_bwd_tc.cu: dQ with rows = queries, dK / dV
 * with rows = keys over query splits whose partials are summed in order -- bit-stable).  fp32 inputs: CUDA-core kernels,
 * dkv is zeroed here and dk / dv accumulate through fp32 atomics (last bits depend on the schedule).
 * ws: dgtd_attention_bwd_ws_floats floats (per-row log-sum-exp and dO.O, plus the split partials). */
int64_t dgtd_attention_bwd_ws_floats(int B, int N, int Nk, int heads);
int dgtd_attention_bwd(const void* q, const void* kv, const void* out, const float* dout, float* dq, float* dkv, float* ws,
                       int dtype, int B, int N, int Nk, int heads, float scale, dgtd_stream_t stream);
/* Backward of Mlp.dwconv + act (cod.py:852-854): x / wT / bias as in dgtd_dwconv3_gelu_fwd, g = dL/d(out) fp32 ->
 * du = g * gelu'(conv3(x) + bias) fp32 (B,h,w,C), dwT (9,C) and dbias (C).  bf16 x with C % 64 == 0: persistent
 * TMA-staged kernel (csrc/dwconv3_tma.cu), per-CTA partial gradients in ws (dgtd_dwconv3_gelu_bwd_ws_floats() floats)
 * summed in a fixed order; otherwise (fp32 x, ws NULL) the pixel-strip kernel with fp32 atomics.  The input gradient is
 * dgtd_dwconv3_fwd(du) with the taps rotated by 180 degrees and a zero bias. */
int64_t dgtd_dwconv3_gelu_bwd_ws_floats(void);
int dgtd_dwconv3_gelu_bwd(const void* x, const float* wT, const float* bias, const float* g, float* du, float* dwT,
                          float* dbias, float* ws, int dtype, int B, int h, int w, int C, dgtd_stream_t stream);

/* ---- structure loss (SURVEY.md 8f-3; cod.cal_loss, cod.py:75-84) ------------------------------------------
 * weit = 1 + 5 |avgpool31x31(gt) - gt| (zero padding, divisor 961); depends on the label only. */
int dgtd_boundary_weight_fwd(const float* gt, float* weit, int planes, int H, int W, dgtd_stream_t stream);
/* loss[0] = mean over planes of wbce + wiou; sums (planes x 4) = (sum w*bce, sum w, I, U) saved for backward */
int dgtd_structure_loss_ws_floats(int planes, int64_t HW);
int dgtd_structure_loss_fwd(const float* preds, const float* gt, const float* weit, float* ws, float* sums, float* loss,
                            int planes, int64_t HW, dgtd_stream_t stream);
int dgtd_structure_loss_bwd(const float* preds, const float* gt, const float* weit, const float* sums,
                            const float* grad_out, float* dpreds, int planes, int64_t HW, dgtd_stream_t stream);

/* SSIM constant of the training loss (cod.py:142-144, SSIM :316-351): out[0] = mean(clamp((1 - SSIM(x, y)) / 2, 0, 1)),
 * x = (emb1 - min) / (max - min + 1e-8) with min / max over the whole (planes, H, W) batch tensor, y = image; 3x3
 * means over reflection-padded windows.  No backward (no parameter upstream).  ws: dgtd_ssim_loss_ws_floats(n). */
int dgtd_ssim_loss_ws_floats(int64_t n);
int dgtd_ssim_loss_fwd(const float* emb1, const float* image, float* ws, float* out, int planes, int H, int W,
                       dgtd_stream_t stream);

/* ---- Hitnet iterative decoder (SURVEY.md 8f-2; cod.py:685-807), NHWC fp32, inference semantics -----------
 * BasicConv2d / CAB convs (cod.py:355-368, 434-451): out[m, n] = prelu(scale[n] * conv(x)[m, n] + shift[n])
 * + residual[m, n]; scale/shift = the folded eval-mode BatchNorm (nullable), prelu = the ONE shared slope of
 * nn.PReLU() (nullable), residual nullable (row pitch ldr).  x / out may be channel slices of wider tensors
 * (pixel pitches ldx / ldo), which is how torch.cat (cod.py:778,785,789,791) is realised.  w packed
 * (Cout, ks*ks*Cin) tap-major; input pixel = o*stride + off + tap, zero outside. */
int dgtd_conv_nhwc_affine_fwd(const float* x, const float* w, const float* scale, const float* shift,
                              const float* prelu, const float* residual, int ldr, float* out, int B, int h, int wd,
                              int Cin, int ldx, int oh, int ow, int Cout, int ldo, int ks, int stride, int off,
                              dgtd_stream_t stream);
/* CALayer / SAM gates (cod.py:413-429, 454-506): fixed-order partial channel sums of x (B, hw, C | pitch ldx)
 * -> partial (B, chunks, C), chunks = dgtd_channel_sums_chunks(hw); then
 * gate[b, o] = sigmoid(sum_j W2[o, j] relu(sum_c W1[j, c] mean[b, c])), W1 (Cr, C), W2 (Co, Cr). */
int dgtd_channel_sums_chunks(int hw);
int dgtd_channel_sums_fwd(const float* x, int ldx, float* partial, int B, int hw, int C, dgtd_stream_t stream);
int dgtd_channel_gate_fwd(const float* partial, int nchunks, int hw, const float* w1, const float* w2, float* gate,
                          int B, int C, int Cr, int Co, dgtd_stream_t stream);
/* out = a * ga[b, c] * sa[b] + b * gb[b, c] * sb[b]  (ga, sa, b, gb, sb nullable): CAB tail `res * y + x`
 * (cod.py:447-450) and the SAM fusion (cod.py:487-503). */
int dgtd_gated_sum_fwd(const float* a, int lda, const float* ga, const float* sa, const float* b, int ldb,
                       const float* gb, const float* sb, float* out, int ldo, int B, int hw, int C,
                       dgtd_stream_t stream);
/* bilinear resize NHWC with pixel pitches, both conventions (nn.Upsample(align_corners=True), cod.py:709,733,737) */
int dgtd_resize_nhwc_ld_fwd(const float* x, int ldx, float* out, int ldo, int B, int h, int w, int C, int oh, int ow,
                            int align_corners, dgtd_stream_t stream);
/* out[row, 0:C] = x[row, 0:C] between tensors of different pixel pitch (the other operand of torch.cat) */
int dgtd_copy_channels_fwd(const float* x, int ldx, float* out, int ldo, int64_t rows, int C, dgtd_stream_t stream);
/* out_CFM / out_SAM (cod.py:710-711,793,803): out[row] (+)= bias[0] + sum_c x[row, c] w[c] */
int dgtd_head1_fwd(const float* x, int ldx, const float* w, const float* bias, float* out, int64_t rows, int C,
                   int accumulate, dgtd_stream_t stream);
/* bf16 mode of the decoder convs: col (B*oh*ow, ks*ks*C) bf16 = im2col of prelu(x) (prelu nullable), the A operand
 * of dgtd_linear_fwd (tcgen05) whose weights carry the folded BatchNorm scale and whose bias is the BN shift. */
int dgtd_im2col_act_fwd(const float* x, int ldx, void* col, const float* prelu, int B, int h, int w, int C, int ks,
                        int stride, int off, int oh, int ow, dgtd_stream_t stream);
/* 3x3 / stride 1 / pad 1 conv of the CABs and conv4 as an implicit tcgen05 GEMM (no im2col in HBM): x (B,h,w,Cp)
 * bf16 from dgtd_cast_pad_act_fwd (= bf16(prelu(x)), channels zero-padded to Cp, a multiple of 64); the A operand
 * of k-block (tap, 64-channel chunk) is ONE 4-D TMA box {64 ch, 16 px, 8 rows} shifted by the tap, zero fill outside
 * the image = the padding; w (Cout, 9*Cp) bf16 tap-major (BatchNorm scale folded in); out (B*h*w, ldo) fp32
 * = conv + bias. */
int dgtd_cast_pad_act_fwd(const float* x, int ldx, void* out, const float* prelu, int64_t rows, int C, int Cp,
                          dgtd_stream_t stream);
int dgtd_conv3x3_tc_fwd(const void* x, const void* w, const float* bias, float* out, int B, int h, int wd, int Cp,
                        int Cout, int ldo, dgtd_stream_t stream);
/* `output.sigmoid()` of the predict mode (cod.py:212,217) */
int dgtd_sigmoid_fwd(const float* x, float* out, int64_t n, dgtd_stream_t stream);

/* ---- training of the Hitnet decoder (SURVEY.md 8f-2 under autograd; csrc/hitnet_train.cu) ------------------------
 * All reductions in a fixed order (per-CTA partials in double + one finalising pass; no atomics).  NHWC fp32 maps,
 * `ld*` = pixel pitch.  ws: scratch of dgtd_col_stats_ws_bytes(M, C) bytes (8-byte aligned).
 * Train-mode nn.BatchNorm2d of BasicConv2d (cod.py:362,366-367): mean / rstd of the batch (biased variance) are
 * written for the backward, out = (y - mean) rstd gamma + beta; run_mean / run_var (nullable together) get the
 * momentum update with the unbiased variance. */
int64_t dgtd_col_stats_ws_bytes(int64_t M, int C);
int dgtd_bn_train_fwd(const float* y, int ldy, const float* gamma, const float* beta, float* run_mean, float* run_var,
                      float momentum, float eps, float* out, int ldo, float* mean, float* rstd, void* ws, int64_t M,
                      int C, dgtd_stream_t stream);
/* the apply step alone with given statistics (eval-mode BatchNorm inside an autograd graph) */
int dgtd_bn_apply_fwd(const float* y, int ldy, const float* mean, const float* rstd, const float* gamma,
                      const float* beta, float* out, int ldo, int64_t M, int C, dgtd_stream_t stream);
/* dgamma = sum dy xhat, dbeta = sum dy; batch_stats 1: dx = gamma rstd (dy - dbeta / M - xhat dgamma / M),
 * 0 (fixed statistics): dx = gamma rstd dy.  y = the conv output the forward normalised. */
int dgtd_bn_train_bwd(const float* dy, int lddy, const float* y, int ldy, const float* mean, const float* rstd,
                      const float* gamma, float* dx, int lddx, float* dgamma, float* dbeta, void* ws, int batch_stats,
                      int64_t M, int C, dgtd_stream_t stream);
/* nn.PReLU() with ONE slope (the `act` every CAB shares, cod.py:686,440): v = u >= 0 ? u : slope u over n values
 * (n % 4 == 0); backward du = g (u >= 0 ? 1 : slope), dslope[0] = sum g u [u < 0]; ws: dgtd_prelu_bwd_ws_bytes(n). */
int dgtd_prelu_fwd(const float* u, const float* slope, float* v, int64_t n, dgtd_stream_t stream);
int64_t dgtd_prelu_bwd_ws_bytes(int64_t n);
int dgtd_prelu_bwd(const float* u, const float* g, const float* slope, float* du, float* dslope, void* ws, int64_t n,
                   dgtd_stream_t stream);
/* partial[b][chunk][c] = sum over the chunk's pixels of a * b (same chunking as dgtd_channel_sums_fwd): the channel
 * dots sum_p g x that the gates' backward starts from. */
int dgtd_channel_dot_fwd(const float* a, int lda, const float* b, int ldb, float* partial, int B, int hw, int C,
                         dgtd_stream_t stream);
/* Backward of out = x * gc[c] * gs, gc = sigmoid(W2 relu(W1 m)) (CALayer cod.py:427-429 / SAM.fc :482), gs =
 * sigmoid(v2 relu(V1 m)) (SAM.fc_wight :480; Cs = 0: no scalar gate), m = mean(x): part = channel sums of x, dpart =
 * channel dots of (g, x).  Writes dmean (B,C) (to be spread as dmean / hw over the pixels) and the weight gradients
 * dw1 (Cr,C), dw2 (C,Cr), dv1 (Cs,C), dv2 (Cs); accumulate 1 adds to them (SAM runs both inputs through the same
 * weights).  One CTA per image + a fixed-order sum over the images; ws: dgtd_gate_bwd_ws_floats(B, C, Cr, Cs) floats. */
int64_t dgtd_gate_bwd_ws_floats(int B, int C, int Cr, int Cs);
int dgtd_gate_bwd(const float* part, int nch, int hw, const float* dpart, int nchd, const float* w1, const float* w2,
                  const float* v1, const float* v2, float* dmean, float* dw1, float* dw2, float* dv1, float* dv2,
                  float* ws, int accumulate, int B, int C, int Cr, int Cs, dgtd_stream_t stream);
/* out = g * gate[b,c] * scal[b] + dmean[b,c] / hw  (scal, dmean nullable): gradient w.r.t. the gated operand */
int dgtd_gated_bwd(const float* g, int ldg, const float* gate, const float* scal, const float* dmean, float* out, int ldo,
                   int B, int hw, int C, dgtd_stream_t stream);
/* backward of dgtd_head1_fwd: dx[row,c] = g[row] w[c] (dx nullable), dw[c] = sum g[row] x[row,c], db[0] = sum g */
int dgtd_head1_bwd(const float* g, const float* x, int ldx, const float* w, float* dx, int lddx, float* dw, float* db,
                   void* ws, int64_t rows, int C, dgtd_stream_t stream);
/* adjoint of dgtd_resize_nhwc_ld_fwd (gather form): g (B,oh,ow,C) -> dx (B,h,w,C) */
int dgtd_resize_nhwc_ld_bwd(const float* g, int ldg, float* dx, int lddx, int B, int h, int w, int C, int oh, int ow,
                            int align_corners, dgtd_stream_t stream);

/* ---- evaluation metrics (SURVEY.md 8f-4; twig/metric/{MAE,Smeasure,Fmeasure,Emeasure}.py:18-36 + pysodmetrics
 * 1.3.1) -- the four evaluators of config/cod.yml:123-128 / sod.yml:85-89.
 * pred, gt (B,1,H,W) fp32 in [0,1] as the `predict` mode returns them (cod.py:217).  Quantises both like the
 * wrappers do (`(x * 255).astype(np.uint8)`, gt > 128), min-max normalises the prediction per image and writes
 * out[b] = {MAE, S-measure (alpha = 0.5)} in float64, from exact integer moments (bit-stable).  curves (nullable):
 * (B, 2, 256) float64 = per image the changeable F-measure (beta^2 = 0.3) and the E-measure at the 256 thresholds
 * (entry i = threshold 255 - i, the library's order), from exact fg / bg histograms of the re-quantised prediction.
 * ws: 256-byte aligned scratch of dgtd_sod_metrics_ws_bytes(B, H, W). */
int64_t dgtd_sod_metrics_ws_bytes(int B, int H, int W);
int dgtd_sod_metrics_fwd(const float* pred, const float* gt, void* ws, double* out, double* curves, int B, int H,
                         int W, dgtd_stream_t stream);
/* weighted F-measure (Margolin et al., CVPR 2014; pysodmetrics 1.3.1 `WeightedFmeasure`, beta = 1): same inputs,
 * quantisation and normalisation as dgtd_sod_metrics_fwd; out[b] = F^w of image b in float64 (0 for an empty ground
 * truth).  Every background pixel takes the error of its nearest foreground pixel under the exact Euclidean distance;
 * among equidistant ones the pixel with the lowest column, then the lowest row, is taken (the choice of
 * scipy.ndimage.distance_transform_edt(return_indices=True)).  Fixed-order reductions: bit-stable, independent of
 * batch composition.  H > 1, W > 1, H * W < 2^28.  ws: 256-byte aligned scratch of dgtd_sod_wfm_ws_bytes(B, H, W). */
int64_t dgtd_sod_wfm_ws_bytes(int B, int H, int W);
int dgtd_sod_wfm_fwd(const float* pred, const float* gt, void* ws, double* out, int B, int H, int W,
                     dgtd_stream_t stream);
/* The same two evaluations for images of different sizes in one padded batch: pred, gt (B,1,Hmax,Wmax), image b in
 * the top-left sizes[b] = (H_b, W_b) of its plane; the rest of the plane is never read.  sizes: device int32 (B, 2)
 * with 2 <= H_b <= Hmax and 2 <= W_b <= Wmax; an image whose size breaks that reads nothing and gets NaN results.
 * Image b's out, curves and F^w are bit-identical to dgtd_sod_metrics_fwd / dgtd_sod_wfm_fwd on its contiguous
 * H_b x W_b crop alone.  ws: dgtd_sod_metrics_ws_bytes(B, Hmax, Wmax) / dgtd_sod_wfm_ws_bytes(B, Hmax, Wmax). */
int dgtd_sod_metrics_sized_fwd(const float* pred, const float* gt, const int32_t* sizes, void* ws, double* out,
                               double* curves, int B, int Hmax, int Wmax, dgtd_stream_t stream);
int dgtd_sod_wfm_sized_fwd(const float* pred, const float* gt, const int32_t* sizes, void* ws, double* out, int B,
                           int Hmax, int Wmax, dgtd_stream_t stream);

/* ---- optimizer step of the training configuration (config/sod.yml:56-76; torch.optim.AdamW semantics) ----------
 * One launch over flat fp32 buffers p, g, m, v (the hot path's gradients already live in one flat buffer,
 * twig/graphs.py).  table: nslices entries of dgtd_adamw_slice_bytes() bytes = {int64 off; int32 n (<= 4096);
 * float lr; float weight_decay; int32 pad} -- one per slice of one parameter, which is how the per-prefix lr
 * multipliers of paramwise_cfg.custom_keys are applied.  g is multiplied by grad_scale first (1 / world size after
 * a sum all-reduce).  step = 1-based step count for the bias corrections.  lr_scale multiplies every slice's lr
 * (the factor of the run's scheduler, e.g. CosineAnnealingLR of config/sod.yml param_scheduler; 1 = constant lr). */
int dgtd_adamw_slice_bytes(void);
int dgtd_adamw_step(float* p, const float* g, float* m, float* v, const void* table, int nslices, float beta1, float beta2,
                    float eps, int step, float grad_scale, float lr_scale, dgtd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DGTD_OPS_H_ */
