/*
 * b200unet — C ABI of the B200-native (sm_100a) U-Net hot path.
 *
 * Drop-in boundary for the hot path of caki35/UNet-Torch (reference = /root/reference):
 *   Model.py:7-169  (DoubleConv / Down / Up / OutConv / UNet.forward)  and
 *   loss.py:215-251, 442-516 (DiceLoss, calc_loss 'dice_bce_mc' / 'CE' / 'mse' / 'mseMC').
 * The reference has no native code; every entry point below replaces the PyTorch library op the
 * reference calls at the cited line. The Python host layer (unet-torch_b200/) binds these with ctypes.
 *
 * Conventions
 *   - All pointers are DEVICE pointers owned by the caller; kernels never allocate or free.
 *   - Activations are NHWC bf16. `*_cs` arguments are the pixel pitch in ELEMENTS (>= channel count), so
 *     a tensor may be a channel slice of a wider buffer (the decoder concat buffer, Model.py:79).
 *   - `stream` is the caller's cudaStream_t. All launches are asynchronous; nothing synchronises.
 *   - Return 0 on success, non-zero on bad shape / alignment / launch failure; text via b200unet_last_error().
 *   - No CPU fallback anywhere: an unsupported shape is an error.
 */
#ifndef B200UNET_H_
#define B200UNET_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* cudaStream_t */

int b200unet_version(void);
const char* b200unet_last_error(void);
/* Number of kernels launched through this library since load (for bench.py's gpu_launches). */
int64_t b200unet_launch_count(void);

/* ---- tile geometry shared with the host (pixel tile of the implicit GEMMs) ------------------------------- */
int b200unet_tile_h(void); /* 8  */
int b200unet_tile_w(void); /* 16 */

/* ---- weight preparation (fp32 master parameters -> bf16 GEMM operands), once per optimizer step ---------- */
/* nn.Conv2d weight OIHW fp32 [K][C][3][3] (Model.py:15-16,19-20) -> fprop operand [K][3][3][C] bf16 and
 * dgrad operand [C][3][3][K] bf16 with the taps rotated by 180 degrees. Either output may be NULL. */
int b200unet_prep_conv3x3_weight(const float* w_oihw, void* w_fprop, void* w_dgrad, int K, int C,
                                 b200_stream_t stream);
/* nn.ConvTranspose2d weight [Cin][Cup][2][2] fp32 (Model.py:56-57) -> fprop operand [(i,j,d)][ci] bf16 and
 * dgrad operand [ci][(i,j,d)] bf16. */
int b200unet_prep_convt2x2_weight(const float* w, void* w_fprop, void* w_dgrad, int Cin, int Cup,
                                  b200_stream_t stream);

/* ---- tensor-core implicit GEMMs (tcgen05 / TMEM / TMA) ---------------------------------------------------- */
/* 3x3, pad 1, no bias (nn.Conv2d, Model.py:15-16,19-20). y[n,h,w,k] = sum_{r,s,c} x[n,h+r-1,w+s-1,c] w[k,r,s,c].
 * Used for fprop (w = fprop operand) and for dgrad (x = dy, w = dgrad operand, Cin/Cout swapped).
 * stats_partial: NULL or fp32 [rows][2][Cout] partial sums and sums of squares of the bf16 outputs, rows =
 * b200unet_conv3x3_stat_rows(N,H,W,Cin,Cout) (one row per pixel tile, or per persistent CTA for the resident-weight
 * kernel used when Cin <= 128); feeds BatchNorm2d (Model.py:17,21) through b200unet_bn_reduce_partials.
 * Requires Cin % 64 == 0 and Cout % 64 == 0. */
int b200unet_conv3x3_stat_rows(int N, int H, int W, int Cin, int Cout);
/* Which of the 3x3 kernels b200unet_conv3x3_igemm picks: each argument -1 = automatic (measured rule), 0 = never,
 * 1 = whenever applicable. resident: persistent resident-weight kernels (Cin <= 128); resident_pairs: their CTA-pair
 * (cta_group::2) form; streaming_pairs: the CTA-pair streaming kernel (Cin >= 256). Test / tuning aid; call
 * b200unet_conv3x3_stat_rows again afterwards (the statistics row count depends on the kernel). */
int b200unet_set_kernel_choice(int resident, int resident_pairs, int streaming_pairs);
int b200unet_conv3x3_igemm(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial,
                           int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* Backward-data launch whose OUTPUT y is the gradient g at the output of a BatchNorm+ReLU (Model.py:17-18 / 21-22 of the layer
 * in front): the first pass of that BatchNorm's backward (b200unet_bn_relu_bwd_reduce) is fused into the epilogue. bn_y = that
 * layer's saved pre-BN tensor (pitch bn_y_cs), scale/shift/mean/rstd its affine and statistics ([Cout] each); partial receives
 * [rows][2][Cout] = (sum da, sum da*xhat) with da = g * [scale*bn_y + shift > 0], rows = b200unet_conv3x3_dgrad_bnred_rows(...)
 * (0 = this shape has no fused form: use b200unet_conv3x3_igemm + b200unet_bn_relu_bwd_reduce). Saves one 4 B/element pass. */
int b200unet_conv3x3_dgrad_bnred_rows(int N, int H, int W, int Cin, int Cout);
int b200unet_conv3x3_igemm_bnred(const void* x, int x_cs, const void* w, void* y, int y_cs, const void* bn_y, int bn_y_cs,
                                 const float* scale, const float* shift, const float* mean, const float* rstd,
                                 float* partial, int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* Eval-mode variant (running statistics, Model.py:17-18 with module.eval()): BatchNorm folded to a per-channel
 * scale/shift ([Cout] fp32 each, 16-byte aligned; b200unet_bn_eval_affine produces them) and applied with the ReLU in the
 * epilogue on the fp32 accumulators: a = bf16(relu(scale * conv(x) + shift)). The pre-BN tensor never reaches HBM. */
int b200unet_conv3x3_bn_relu_igemm(const void* x, int x_cs, const void* w, const float* scale, const float* shift, void* a,
                                   int a_cs, int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* ConvTranspose2d(Cin, Cup, 2, 2) + bias (Model.py:56-57,66): out[n,2h+i,2w+j,d] = b[d] + sum_c x[n,h,w,c] W[c,d,i,j],
 * written with pitch out_cs into a (H2 x W2) canvas at row/col offset (pad_top, pad_left) (F.pad, Model.py:69-73). */
int b200unet_convt2x2_fprop(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs,
                            int N, int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left,
                            b200_stream_t stream);
/* its backward-data: dx[n,h,w,c] = sum_{d,i,j} du[n,2h+i,2w+j,d] W[c,d,i,j]. */
int b200unet_convt2x2_dgrad(const void* du, int du_cs, const void* w_dgrad, void* dx, int dx_cs, int N, int H,
                            int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left,
                            b200_stream_t stream);

/* Weight gradients. partial = fp32 workspace of b200unet_wgrad_workspace_floats() floats; dw = fp32 gradient in
 * the PARAMETER's own layout (OIHW for conv, [Cin][Cup][2][2] for convT), overwritten (not accumulated). */
int64_t b200unet_conv3x3_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cout);
int b200unet_conv3x3_wgrad(const void* x, int x_cs, const void* dy, int dy_cs, float* partial, float* dw_oihw,
                           int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
int64_t b200unet_convt2x2_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cup);
int b200unet_convt2x2_wgrad(const void* x, int x_cs, const void* du, int du_cs, float* partial, float* dw,
                            int N, int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left,
                            b200_stream_t stream);

/* ---- inc.conv1 on the tensor cores (Model.py:111 -> :15-16 with Cin = n_channels <= 7) ------------------- */
/* x fp32 NCHW [N][Cin][H][W] -> col bf16 NHWC [N][H][W][64] (pitch col_cs): col[..., c*9+r*3+s] = x[n,c,h+r-1,w+s-1],
 * zero outside the image and in columns >= 9*Cin. */
int b200unet_first_im2col(const float* x_nchw, void* col, int col_cs, int N, int H, int W, int Cin,
                          b200_stream_t stream);
/* nn.Conv2d weight OIHW fp32 [Cout][Cin][3][3] -> bf16 [Cout][64] operand matching the im2col columns. */
int b200unet_prep_first_weight(const float* w_oihw, void* w1, int Cout, int Cin, b200_stream_t stream);
/* inc.conv1 (Model.py:111 -> :15-16) FUSED: y = conv3x3(x) straight from the fp32 NCHW network input; the im2col rows are
 * built in shared memory inside the tcgen05 GEMM kernel, no im2col tensor reaches HBM. w1 = b200unet_prep_first_weight's
 * [Cout][64] bf16 operand; stats_partial as b200unet_conv1x1_c64_igemm (rows = b200unet_conv1x1_c64_stat_rows). Cin <= 7. */
int b200unet_conv3x3_first_igemm(const float* x_nchw, const void* w1, void* y, int y_cs, float* stats_partial, int N, int H,
                                 int W, int Cin, int Cout, b200_stream_t stream);
/* its eval-mode form: a = bf16(relu(scale * conv + shift)) */
int b200unet_conv3x3_first_bn_relu_igemm(const float* x_nchw, const void* w1, const float* scale, const float* shift,
                                         void* a, int a_cs, int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* and its weight gradient dw (fp32 OIHW [Cout][Cin][3][3]) from x and dy, im2col rows again built in shared memory */
int64_t b200unet_conv3x3_first_tc_wgrad_workspace_floats(int N, int H, int W, int Cout);
int b200unet_conv3x3_first_tc_wgrad(const float* x_nchw, const void* dy, int dy_cs, float* partial, float* dw_oihw, int N,
                                    int H, int W, int Cin, int Cout, b200_stream_t stream);
/* y[n,h,w,k] = sum_j x[n,h,w,j] w[k,j], j < 64 (1x1 convolution of a 64-channel tensor; tcgen05, persistent CTAs,
 * weights resident). stats_partial as for b200unet_conv3x3_igemm with rows = b200unet_conv1x1_c64_stat_rows(). */
int b200unet_conv1x1_c64_stat_rows(int N, int H, int W, int Cout);
int b200unet_conv1x1_c64_igemm(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial,
                               int N, int H, int W, int Cout, b200_stream_t stream);
int b200unet_conv1x1_c64_bn_relu_igemm(const void* x, int x_cs, const void* w, const float* scale, const float* shift, void* a,
                                       int a_cs, int N, int H, int W, int Cout, b200_stream_t stream);
/* dw[k][j] = sum_{n,h,w} dy[n,h,w,k] col[n,h,w,j] for j < T (T = 9*Cin): inc.conv1's weight gradient, written as
 * fp32 OIHW [Cout][Cin][3][3] (= [Cout][T]). partial: b200unet_conv1x1_c64_wgrad_workspace_floats() floats. */
int64_t b200unet_conv1x1_c64_wgrad_workspace_floats(int N, int H, int W, int Cout);
int b200unet_conv1x1_c64_wgrad(const void* col, int col_cs, const void* dy, int dy_cs, float* partial, float* dw,
                               int N, int H, int W, int T, int Cout, b200_stream_t stream);

/* ---- 1x1 convolutions of the attention gates (Attention_block W_q / W_x, Model.py:260-275) ------------------ */
/* nn.Conv2d(Cin, Cout, 1) + bias as a tcgen05 GEMM over NHWC bf16: y[n,h,w,k] = b[k] + sum_c x[n,h,w,c] w[k][c], w bf16
 * [Cout][Cin]. Also its backward-data (x = dy, w = the transposed operand [Cin][Cout], bias NULL). stats_partial: NULL or
 * fp32 [b200unet_conv1x1_stat_rows][2][stat_channels] sums / sums of squares of the first stat_channels <= Cout channels of
 * the bf16 outputs (feeds the BatchNorm2d that follows, Model.py:263,272). Requires Cin % 64 == 0 and Cout % 64 == 0 (the host pads a 32-channel gate with zero weights). */
int b200unet_conv1x1_stat_rows(int N, int H, int W);
int b200unet_conv1x1_fprop(const void* x, int x_cs, const void* w, const float* bias, void* y, int y_cs, float* stats_partial,
                           int stat_channels, int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* dw[k][c] = sum_{n,h,w} dy[n,h,w,k] x[n,h,w,c] for k < Cout_real, fp32 [Cout_real][Cin] (= the OIHW gradient). */
int64_t b200unet_conv1x1_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cout);
int b200unet_conv1x1_wgrad(const void* x, int x_cs, const void* dy, int dy_cs, float* partial, float* dw, int N, int H, int W,
                           int Cin, int Cout, int Cout_real, b200_stream_t stream);
/* b200unet_convt2x2_fprop with the BatchNorm statistics of its output: stats_partial fp32
 * [b200unet_convt2x2_stat_rows][2][stat_channels] (the first stat_channels <= Cup channels). The gate's `up` followed by W_q (Model.py:287-288) is ONE ConvTranspose2d with the
 * composed weight, so the C_q-channel upsampled map never exists. */
int b200unet_convt2x2_stat_rows(int N, int H, int W);
int b200unet_convt2x2_fprop_stats(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs,
                                  float* stats_partial, int stat_channels, int N, int H, int W, int Cin, int Cup, int H2,
                                  int W2, int pad_top, int pad_left, b200_stream_t stream);

/* ---- attention gate, bandwidth-bound part (Attention_block.forward, Model.py:286-296) ----------------------------
 * q1 / x1: the pre-BatchNorm maps W_q(up(q)) and W_x(x), NHWC bf16 with C real channels (32, 64, 128 or 256) and pitches
 * q1_cs / x1_cs; scale_* / shift_*: the BatchNorm affine of each ([C] fp32); w_psi [C], b_psi [1]: the psi convolution.
 * E = relu(Q1 + X1) and A are never stored; s (fp32, one value per pixel) is psi's output before its BatchNorm2d(1). */
int64_t b200unet_gate_workspace_floats(int C);
int b200unet_gate_stat_rows(int64_t pixels, int C);
/* s = b_psi + sum_c w_psi[c] * relu(scale_q*q1 + shift_q + scale_x*x1 + shift_x)[c]; stats_partial: NULL or fp32
 * [b200unet_gate_stat_rows][2] (sum s, sum s^2) for BatchNorm2d(1) (Model.py:280). */
int b200unet_gate_psi_fwd(const void* q1, int q1_cs, const void* x1, int x1_cs, const float* scale_q, const float* shift_q,
                          const float* scale_x, const float* shift_x, const float* w_psi, const float* b_psi, float* s,
                          float* stats_partial, int64_t pixels, int C, b200_stream_t stream);
/* out = x * sigmoid(scale_p * s + shift_p) over Cx channels (Model.py:295-296); out may be a channel slice (concat buffer). */
int b200unet_gate_apply_fwd(const void* x, int x_cs, const float* s, const float* scale_p, const float* shift_p, void* out,
                            int out_cs, int64_t pixels, int Cx, b200_stream_t stream);
/* Backward of the product: A = sigmoid(scale_p*s + shift_p); dx = g * A (bf16; NULL = not written, see b200unet_gate_dx);
 * dz = (sum_c g*x) * A * (1 - A) (fp32, one per pixel); sums2 = fp64 [sum dz, sum dz * shat] with shat = (s - mean_p) * rstd_p
 * (BatchNorm2d(1) backward). */
int b200unet_gate_apply_bwd(const void* g, int g_cs, const void* x, int x_cs, const float* s, const float* scale_p,
                            const float* shift_p, const float* mean_p, const float* rstd_p, void* dx, int dx_cs, float* dz,
                            float* workspace, double* sums2, int64_t pixels, int Cx, b200_stream_t stream);
/* dx <- g * A + dx in place: the product's gradient added to the W_x backward-data already in dx (one pass instead of a store in
 * b200unet_gate_apply_bwd plus a separate add). */
int b200unet_gate_dx(const void* g, int g_cs, const float* s, const float* scale_p, const float* shift_p, void* dx, int dx_cs,
                     int64_t pixels, int Cx, b200_stream_t stream);
/* ds = BatchNorm2d(1) backward of dz (sums2 = the, under SyncBN all-reduced, sums above; count = pixels per channel);
 * dE = ds * w_psi * [E > 0]. sums fp64 [4C + 8]: [0,C) sum dE, [C,2C) sum dE*Qhat, [2C,3C) sum dE*Xhat, [3C,4C) sum ds*E,
 * [4C] sum ds. */
int b200unet_gate_bwd_reduce(const void* q1, int q1_cs, const void* x1, int x1_cs, const float* scale_q, const float* shift_q,
                             const float* scale_x, const float* shift_x, const float* mean_q, const float* rstd_q,
                             const float* mean_x, const float* rstd_x, const float* w_psi, const float* s, const float* dz,
                             const float* gamma_p, const float* mean_p, const float* rstd_p, const double* sums2, double count,
                             float* ds, float* workspace, double* sums, int64_t pixels, int C, b200_stream_t stream);
/* q1 <- BN_q backward of dE, x1 <- BN_x backward of dE (bf16, in place); parameter gradients from sums_local (NULL = sums)
 * and sums2_local; dbias fp32 [2C] = per-channel sums of the two stored gradients (the bias gradients of the two convs). */
int b200unet_gate_bwd_apply(void* q1, int q1_cs, void* x1, int x1_cs, const float* scale_q, const float* shift_q,
                            const float* scale_x, const float* shift_x, const float* gamma_q, const float* mean_q,
                            const float* rstd_q, const float* gamma_x, const float* mean_x, const float* rstd_x,
                            const float* w_psi, const float* ds, const double* sums, const double* sums_local,
                            const double* sums2_local, double count, float* dgamma_q, float* dbeta_q, float* dgamma_x,
                            float* dbeta_x, float* dw_psi, float* db_psi, float* dgamma_p, float* dbeta_p, float* workspace,
                            float* dbias, int64_t pixels, int C, b200_stream_t stream);
/* C[z][m][n] (+)= sum_k A[z][m][k] B[z][k][n] (+ bias_m[m]), fp32, arbitrary ELEMENT strides (am, ak, ...; az/bz/cz between
 * batch entries). Weight-side algebra of the gates: W'[c,h,i,j] = sum_d W_up[c,d,i,j] W_q[h,d] and its backward. */
int b200unet_sgemm_strided(const float* A, const float* B, float* C, const float* bias_m, int M, int N, int K, int64_t am,
                           int64_t ak, int64_t bk, int64_t bn, int64_t cm, int64_t cn, int batch, int64_t az, int64_t bz,
                           int64_t cz, int accumulate, b200_stream_t stream);

/* out[i] = sum_b part[b][i], b < batches, i < n (fixed order): joins batch-parallel partial products of the call above. */
int b200unet_sum_batches(const float* part, float* out, int64_t n, int batches, b200_stream_t stream);

/* ---- first layer and head (tiny channel counts: bandwidth-bound CUDA-core kernels) ------------------------ */
/* inc.conv1: x fp32 NCHW [N][Cin<=4][H][W] (Trainer.py:700-702 hands fp32 NCHW) -> y bf16 NHWC [..][Cout] + stats. */
int b200unet_conv3x3_first_fprop(const float* x_nchw, const float* w_oihw, void* y, int y_cs, float* stats_partial,
                                 int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
int64_t b200unet_conv3x3_first_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cout);
int b200unet_conv3x3_first_wgrad(const float* x_nchw, const void* dy, int dy_cs, float* partial, float* dw_oihw,
                                 int N, int H, int W, int Cin, int Cout, b200_stream_t stream);
/* OutConv 1x1 + bias (Model.py:86-92): a bf16 NHWC [..][Cin] -> logits fp32 NCHW [N][ncls][H][W]. ncls <= 8. */
int b200unet_head_fprop(const void* a, int a_cs, const float* w, const float* bias, float* logits_nchw, int N,
                        int H, int W, int Cin, int ncls, b200_stream_t stream);
/* backward: dz fp32 NCHW -> da bf16 NHWC, dw fp32 [ncls][Cin], db fp32 [ncls]. partial: workspace. */
int64_t b200unet_head_bwd_workspace_floats(int N, int H, int W, int Cin, int ncls);
int b200unet_head_bwd(const float* dz_nchw, const void* a, int a_cs, const float* w, void* da, int da_cs,
                      float* partial, float* dw, float* db, int N, int H, int W, int Cin, int ncls,
                      b200_stream_t stream);
/* The same head for 1 <= ncls <= 256 (head_many.cu), Cin 64 or 128: classes in compile-time chunks of 8, so one kernel
 * serves every count; at ncls <= 8 the logits are bit-identical to b200unet_head_fprop, which stays faster there.
 * Backward: da bf16 NHWC, dw fp32 [ncls][Cin], db fp32 [ncls], reduced in a fixed order (fp64) from per-block partials in
 * `partial` (b200unet_head_many_bwd_workspace_floats floats). */
int b200unet_head_many_fprop(const void* a, int a_cs, const float* w, const float* bias, float* logits_nchw, int N,
                             int H, int W, int Cin, int ncls, b200_stream_t stream);
int64_t b200unet_head_many_bwd_workspace_floats(int N, int H, int W, int Cin, int ncls);
int b200unet_head_many_bwd(const float* dz_nchw, const void* a, int a_cs, const float* w, void* da, int da_cs,
                           float* partial, float* dw, float* db, int N, int H, int W, int Cin, int ncls,
                           b200_stream_t stream);

/* ---- BatchNorm2d + ReLU (+ MaxPool2d(2)) bandwidth kernels (Model.py:17-18,21-22,36,42) ------------------- */
/* Reduce the per-tile partials of the conv epilogue into batch statistics and the affine (scale, shift):
 *   sums[0..C)   = sum y, sums[C..2C) = sum y^2 (fp64, so SyncBN can all-reduce them between the two calls). */
int b200unet_bn_reduce_partials(const float* stats_partial, int64_t mtiles, int C, double* sums,
                                b200_stream_t stream);
/* Pre-reduction of statistics rows: out[b][col] = sum of partial[r][col] over r = b (mod out_rows), fixed order. For epilogues
 * that emit one row per pixel tile (the attention gates' GEMMs: up to 131 072 rows) ahead of the one-block-per-32-channels
 * finalisation kernels. ncols = 2 * C: a power of two <= 256 or a multiple of 256. */
int b200unet_fold_rows(const float* partial, int64_t rows, int ncols, float* out, int out_rows, b200_stream_t stream);
/* count = number of elements per channel behind `sums` (global count under SyncBN). Writes mean/rstd (saved for
 * backward), scale = gamma*rstd, shift = beta - mean*scale; if running_mean != NULL also
 * running_mean = (1-mom)*rm + mom*mean, running_var = (1-mom)*rv + mom*var*count/(count-1). */
int b200unet_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, float* mean, float* rstd,
                         float* scale, float* shift, int C, b200_stream_t stream);
/* The two calls above in ONE launch for the single-GPU forward (no cross-rank step in between): reduces the partial rows in
 * a fixed order (fp64) and finalises; num_batches_tracked (int64 scalar, may be NULL) is incremented on the device. */
int b200unet_bn_reduce_finalize(const float* stats_partial, int64_t rows, int C, double count, const float* gamma,
                                const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                                int64_t* num_batches_tracked, float* mean, float* rstd, float* scale, float* shift,
                                b200_stream_t stream);
/* eval mode: scale/shift from running statistics. */
int b200unet_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                            const float* running_var, float eps, float* scale, float* shift, int C,
                            b200_stream_t stream);
/* eval mode WITH autograd (frozen-BatchNorm fine-tuning, saliency maps): mean = running_mean, rstd = rsqrt(running_var +
 * eps) in the form the backward kernels take. With these and an all-zero `sums` vector, b200unet_bn_relu_bwd_apply
 * computes the running-statistics backward dy = gamma * rstd * da; dgamma / dbeta come from `sums_local`. */
int b200unet_bn_eval_stats(const float* running_mean, const float* running_var, float eps, float* mean, float* rstd, int C,
                           b200_stream_t stream);
/* a = relu(scale*y + shift) written with pitch a_cs (possibly into the concat buffer). If pooled != NULL also
 * writes the 2x2/2 max-pooled tensor [N][H/2][W/2][C] (pitch C) and, if pool_idx != NULL, the window position
 * 0..3 (= 2*dh + dw, first maximum in row-major order, NaN wins: nn.MaxPool2d semantics) as uint8. */
int b200unet_bn_relu_fwd(const void* y, int y_cs, const float* scale, const float* shift, void* a, int a_cs,
                         void* pooled, uint8_t* pool_idx, int N, int H, int W, int C, b200_stream_t stream);
/* Backward of (BN -> ReLU [-> skip + pool]). g1 = gradient w.r.t. a arriving with pitch g1_cs (may be NULL if
 * pooled-only); g_pool/pool_idx = gradient w.r.t. the pooled tensor (NULL if the layer is not pooled).
 * Pass 1 (reduce): per-block partial sums of da and da*xhat where da = (g1 + unpool(g_pool)) * [a > 0]. */
int64_t b200unet_bn_bwd_workspace_floats(int N, int H, int W, int C);
/* (b200unet_bn_relu_bwd_reduce_rows: pass 1 only - leaves the block partials [*rows_out][2][C] in `partial` for a fused
 * cross-rank reduction, b200unet_nvl_rows_allreduce) */
int b200unet_bn_relu_bwd_reduce_rows(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                     int y_cs, const float* scale, const float* shift, const float* mean,
                                     const float* rstd, float* partial, int* rows_out, int N, int H, int W, int C,
                                     b200_stream_t stream);
int b200unet_bn_relu_bwd_reduce(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx,
                                const void* y, int y_cs, const float* scale, const float* shift, const float* mean,
                                const float* rstd, float* partial, double* sums, int N, int H, int W, int C,
                                b200_stream_t stream);
/* Pass 2 (apply): dy = gamma*rstd*(da - sum(da)/count - xhat*sum(da*xhat)/count); also dgamma = sums[C..2C),
 * dbeta = sums[0..C) (local sums; `sums` may have been all-reduced for SyncBN, then pass local copies in
 * sums_local for the parameter gradients). */
int b200unet_bn_relu_bwd_apply(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx,
                               const void* y, int y_cs, const float* gamma, const float* scale, const float* shift,
                               const float* mean, const float* rstd, const double* sums, double count,
                               const double* sums_local, void* dy, int dy_cs, float* dgamma, float* dbeta, int N,
                               int H, int W, int C, b200_stream_t stream);
/* out[c] = sum_r partial[r][col_lo + c], c < n: per-channel sums from the [rows][row_pitch] statistics rows a conv
 * epilogue wrote (row_pitch = 2*Cout; columns [0,Cout) hold the sums). Used for the ConvTranspose2d bias gradient
 * (Model.py:56): db = sum over pixels of the upsampled half of the concat gradient. */
int b200unet_partial_colsum(const float* partial, int64_t rows, int row_pitch, int col_lo, int n, float* out,
                            b200_stream_t stream);
/* per-channel sum over pixels of a bf16 NHWC tensor (ConvTranspose2d bias gradient). */
/* nn.MaxPool2d(2) alone (Model.py:36,42) on an NHWC bf16 tensor: first maximum in row-major window order, NaN wins;
 * pool_idx (nullable): window position 0..3 per pooled element ([N][H/2][W/2][C] bytes). Inference path: BatchNorm + ReLU
 * already ran in the conv epilogue (b200unet_conv3x3_bn_relu_igemm). */
int b200unet_maxpool2x2_fwd(const void* a, int a_cs, void* pooled, int p_cs, uint8_t* pool_idx, int N, int H, int W, int C,
                            b200_stream_t stream);
/* Two decoders over one encoder (UNet_multitask, Model.py:172-250): copy a channel slice of an NHWC bf16 buffer into another
 * (the skip half of the second decoder's concat buffer), and out = a + b over channel slices (sum of the two decoders'
 * gradients; out may alias a). Pitches in elements, multiples of 8. */
int b200unet_nhwc_copy(const void* src, int src_cs, void* dst, int dst_cs, int64_t pixels, int C, b200_stream_t stream);
int b200unet_nhwc_add(const void* a, int a_cs, const void* b, int b_cs, void* out, int out_cs, int64_t pixels, int C,
                      b200_stream_t stream);
int64_t b200unet_channel_sum_workspace_floats(int C);
int b200unet_channel_sum(const void* x, int x_cs, float* workspace, float* out, int64_t pixels, int C,
                         b200_stream_t stream);

/* ---- nn.Dropout (Model.py:34-39 after the pooling of Down, :80-81 after the concat of Up) ------------------------- */
/* In place over channels [c_lo, c_lo + nc) of a site tensor [N][H][W][C_site]; x points at channel c_lo of pixel 0, pixel
 * pitch x_cs. For the site element e = ((n*H + h)*W + w)*C_site + c:
 *   (r0..r3) = Philox4x32-10(counter = (lo32(e/4), hi32(e/4), site, 0), key = (lo32(*seed), hi32(*seed)))
 *   x = r[e % 4] < threshold ? bf16(float(x) * scale) : 0
 * threshold in [0, 2^32), scale: the caller's 1/(1-p). The mask depends on (seed, site, e) only, so forward and backward
 * call this with the same arguments. seed: one int64 on the device (no host read: the launch may be captured in a graph).
 * partial (nullable): per-block sums of the OUTPUT channels [sum_lo, sum_lo + sum_n) of the slice, [rows][sum_n] fp32 with
 * rows = b200unet_dropout_partial_rows(N, H, W, nc); reduce with b200unet_partial_colsum(partial, rows, sum_n, 0, sum_n, out)
 * (the ConvTranspose2d bias gradient of a dropped concat gradient). Requires nc and x_cs multiples of 8, x 16-byte aligned,
 * and nc <= 2048 when partial != NULL. */
int b200unet_dropout_partial_rows(int N, int H, int W, int nc);
int b200unet_dropout_mul(void* x, int x_cs, int N, int H, int W, int C_site, int c_lo, int nc, int site, const int64_t* seed,
                         int64_t threshold, float scale, float* partial, int sum_lo, int sum_n, b200_stream_t stream);

/* ---- losses (loss.py:442-516) ----------------------------------------------------------------------------- */
/* 'dice_bce_mc' (loss.py:488-500) and 'CE' (loss.py:468-469) forward, any ncls >= 1. logits fp32 NCHW, target fp32 [N][H][W]
 * (class index stored as float, as the reference DataLoader produces). sums: fp64 scratch of
 * b200unet_loss_sums_doubles() doubles ([sum CE, I_c, Z_c, Y_c], one scalar per 128-byte line), handed unchanged to
 * the backward. loss_out[0] = total loss, [1] = CE, [2] = Dice. mode: 0 = 0.5*CE+0.5*Dice, 1 = CE only.
 * err_flag: set to 1 if a target is outside [0, ncls) (the reference raises). */
int b200unet_loss_sums_doubles(void);
/* `sums` size for a class count: b200unet_loss_sums_doubles() up to 8 classes; past 8 the layout is [CE, I[ncls], Z[ncls],
 * Y[ncls]], the backward's per-class Dice coefficients, then the forward's per-block rows (the per-class sums are reduced
 * in a fixed order). */
int64_t b200unet_loss_sums_doubles_n(int ncls);
/* The leading doubles of `sums` that b200unet_loss_ce_dice_bwd reads: past 8 classes the rest is forward-only scratch, so a
 * caller that keeps `sums` until the backward may keep just this prefix. */
int64_t b200unet_loss_sums_saved_doubles_n(int ncls);
int b200unet_loss_ce_dice_fwd(const float* logits, const float* target, double* sums, float* loss_out,
                              int* err_flag, int N, int ncls, int64_t HW, int mode, b200_stream_t stream);
/* dlogits = grad_out[0] * dL/dlogits. */
int b200unet_loss_ce_dice_bwd(const float* logits, const float* target, const double* sums, const float* grad_out,
                              float* dlogits, int N, int ncls, int64_t HW, int mode, b200_stream_t stream);
/* 'mse' / 'mseMC' (loss.py:473-476): mean((pred - target)^2) over n elements; relu_input != 0 fuses the
 * Trainer's F.relu (Trainer.py:709-710) when the caller wants it (pred = max(o, 0)). */
int b200unet_mse_fwd(const float* pred, const float* target, double* sum, float* loss_out, int64_t n,
                     int relu_input, b200_stream_t stream);
int b200unet_mse_bwd(const float* pred, const float* target, const float* grad_out, float* dpred, int64_t n,
                     int relu_input, b200_stream_t stream);

/* ---- inference head (test_mc3serousv5.py:880-881): fp32 softmax over classes, then first-maximum argmax (any ncls) */
int b200unet_softmax_argmax(const float* logits, int64_t* mask, int N, int ncls, int64_t HW, b200_stream_t stream);

/* ---- the steps either side of the network (edge.cu; SURVEY.md 8f ranks 3 and 4) ------------------------------------ */
/* Input edge (DataLoader.py:661-671, test_mc3serousv5.py:115-125): uint8 images [N][H][W][C] (C <= 4, BGR order as
 * cv2.imread returns) -> fp32 NCHW, each image/channel z-normalised with its own mean and (population) standard
 * deviation over H*W computed exactly (integer sums, fp64 finalisation like numpy); reverse_channels = BGR -> RGB.
 * workspace: b200unet_znorm_workspace_bytes(N, C) bytes. */
int64_t b200unet_znorm_workspace_bytes(int N, int C);
int b200unet_znorm_to_chw(const uint8_t* img_nhwc, void* workspace, float* out_nchw, int N, int H, int W, int C,
                          int reverse_channels, b200_stream_t stream);
/* Inference epilogue (test_mc3serousv5.py:879-887): OutConv + softmax(dim=1) + argmax(dim=1) + np.uint8 in one pass over the
 * last activation (NHWC bf16); bit-identical to b200unet_head_fprop followed by b200unet_softmax_argmax. */
int b200unet_head_mask(const void* a, int a_cs, const float* w, const float* bias, uint8_t* mask, int N, int H, int W,
                       int Cin, int ncls, b200_stream_t stream);
/* Binary-mask epilogue (test.py:393-399): OutConv channel 0 + torch.sigmoid (fp32) + `>= threshold` (0.5) -> {0,1} uint8. */
int b200unet_head_sigmoid_mask(const void* a, int a_cs, const float* w, const float* bias, uint8_t* mask, int N, int H, int W,
                               int Cin, int ncls, float threshold, b200_stream_t stream);
/* Density-map epilogue (test_mc3serousv5.py:961-974): OutConv + F.relu + fp32 division by `divisor` (200 in the
 * reference; 1 = plain F.relu(model(x))) -> fp32 NCHW maps; counts (nullable): [N][ncls] fp64 sums of the stored maps. */
int b200unet_head_density(const void* a, int a_cs, const float* w, const float* bias, float* out_nchw, double* counts,
                          int N, int H, int W, int Cin, int ncls, float divisor, b200_stream_t stream);
/* b200unet_head_mask / b200unet_head_density for 1 <= ncls <= 256 and Cin 64 or 128 (head_many.cu): the mask equals
 * b200unet_head_many_fprop followed by b200unet_softmax_argmax, the maps equal F.relu(logits) / divisor of its logits. */
int b200unet_head_many_mask(const void* a, int a_cs, const float* w, const float* bias, uint8_t* mask, int N, int H, int W,
                            int Cin, int ncls, b200_stream_t stream);
int b200unet_head_many_density(const void* a, int a_cs, const float* w, const float* bias, float* out_nchw, double* counts,
                               int N, int H, int W, int Cin, int ncls, float divisor, b200_stream_t stream);

/* ---- SyncBN over NVLink peer memory (nvl_sync.cu; SURVEY.md 8e): one-shot all-reduce of a small fp64 vector through
 * symmetric buffers mapped into every rank (peer_bufs = HOST array of `world` device pointers, index = rank; each
 * buffer b200unet_nvl_buffer_bytes() bytes, zeroed once before first use), optionally fused with the BatchNorm
 * finalisation of b200unet_bn_finalize. `seq` = 1, 2, 3, ... must advance identically on all ranks; `seq` = 0 takes the
 * next number from a counter inside the rank's own buffer (a launch captured in a CUDA graph then stays valid on replay);
 * do not mix the two numberings on one buffer. One kernel per rank; it spins (bounded) until every peer has published,
 * so each rank must run on its own GPU. */
int64_t b200unet_nvl_buffer_bytes(void);
int b200unet_nvl_allreduce_f64(const double* local, double* out, int n, void* const* peer_bufs, int world, int rank,
                               int64_t seq, b200_stream_t stream);
int b200unet_nvl_bn_sync_finalize(const double* local_sums, double* global_sums, void* const* peer_bufs, int world,
                                  int rank, int64_t seq, double global_count, const float* gamma, const float* beta,
                                  float eps, float momentum, float* running_mean, float* running_var, float* mean,
                                  float* rstd, float* scale, float* shift, int C, b200_stream_t stream);
/* The fast path of both: take the UNREDUCED partial rows [rows][2][C] (conv epilogue statistics, or the block partials of
 * b200unet_bn_relu_bwd_reduce_rows), reduce them, exchange them over NVLink and (forward) finalise BatchNorm in ONE
 * multi-block kernel (one block per 32 channels, each with its own device-side sequence counter: graph-replayable).
 * C <= 2048. sums_local / sums_global: fp64 [2C] each, either may be NULL. */
int b200unet_nvl_rows_allreduce(const float* partial, int64_t rows, int C, void* const* peer_bufs, int world, int rank,
                                double* sums_local, double* sums_global, b200_stream_t stream);
int b200unet_nvl_bn_rows_sync_finalize(const float* stats_partial, int64_t rows, int C, void* const* peer_bufs, int world,
                                       int rank, double global_count, const float* gamma, const float* beta, float eps,
                                       float momentum, float* running_mean, float* running_var,
                                       int64_t* num_batches_tracked, float* mean, float* rstd, float* scale, float* shift,
                                       b200_stream_t stream);
/* Bound on the wait for a peer inside the kernels above (default 600 000 ms, like NCCL's watchdog; 0 = wait forever).
 * On expiry the kernel records the failure in its own buffer, writes NaN to its outputs and returns - it does not trap. */
int b200unet_nvl_set_timeout_ms(int64_t ms);
/* Host read (synchronises `stream`) of this rank's buffer: out3 = {reductions issued through the device-side counter,
 * sequence number of the first reduction that timed out (0 = none), bit mask of the ranks that never arrived}. */
int b200unet_nvl_status(const void* my_buffer, b200_stream_t stream, int64_t* out3);

/* ---- generic fp32 path (generic_f32.cu): check mode and the slow-but-correct route for shapes outside the
 * tensor-core path (H, W not divisible by 16 -> F.pad branch Model.py:69-73 and floor-mode pooling; widths that are not
 * multiples of 64; dropout variants Model.py:34-39,81-82). NCHW fp32 like the reference; `*_ns` = batch stride in
 * elements so that a channel range of the concat tensor is a valid view. One thread per output, fp64 reductions. */
int b200unet_gen_conv3x3(const float* in, int64_t in_ns, const float* w, float* out, int64_t out_ns, int N, int Ci,
    int Co, int H, int W, int transposed, b200_stream_t stream);
int b200unet_gen_conv3x3_wgrad(const float* x, int64_t x_ns, const float* dy, int64_t dy_ns, float* dw, int N, int
    Ci, int Co, int H, int W, b200_stream_t stream);
int b200unet_gen_channel_stats(const float* y, int64_t y_ns, double* sums, int N, int C, int HW, b200_stream_t
    stream);
int b200unet_gen_bn_relu_fwd(const float* y, int64_t y_ns, const float* scale, const float* shift, float* a,
    int64_t a_ns, int N, int C, int HW, b200_stream_t stream);
int b200unet_gen_maxpool2x2(const float* a, int64_t a_ns, float* pooled, uint8_t* idx, int N, int C, int H, int W,
    b200_stream_t stream);
int b200unet_gen_unpool_add(const float* g_pooled, const uint8_t* idx, float* g, int64_t g_ns, int N, int C, int H,
    int W, b200_stream_t stream);
int b200unet_gen_bn_relu_bwd_reduce(const float* g, int64_t g_ns, const float* y, int64_t y_ns, const float* scale,
    const float* shift, const float* mean, const float* rstd, double* sums, int N, int C, int HW, b200_stream_t
    stream);
int b200unet_gen_bn_relu_bwd_apply(const float* g, int64_t g_ns, const float* y, int64_t y_ns, const float* gamma,
    const float* scale, const float* shift, const float* mean, const float* rstd, const double* sums, double count,
    const double* sums_local, float* dy, int64_t dy_ns, float* dgamma, float* dbeta, int N, int C, int HW,
    b200_stream_t stream);
int b200unet_gen_convt2x2_fprop(const float* x, int64_t x_ns, const float* w, const float* bias, float* out,
    int64_t out_ns, int N, int Cin, int Cup, int H, int W, int H2, int W2, int pad_top, int pad_left, b200_stream_t
    stream);
int b200unet_gen_convt2x2_dgrad(const float* du, int64_t du_ns, const float* w, float* dx, int64_t dx_ns, int N,
    int Cin, int Cup, int H, int W, int H2, int W2, int pad_top, int pad_left, b200_stream_t stream);
int b200unet_gen_convt2x2_wgrad(const float* x, int64_t x_ns, const float* du, int64_t du_ns, float* dw, float* db,
    int N, int Cin, int Cup, int H, int W, int H2, int W2, int pad_top, int pad_left, b200_stream_t stream);
int b200unet_gen_conv1x1_fwd(const float* a, int64_t a_ns, const float* w, const float* bias, float* z, int N, int
    C, int J, int64_t HW, b200_stream_t stream);
int b200unet_gen_conv1x1_bwd(const float* dz, const float* a, int64_t a_ns, const float* w, float* da, int64_t
    da_ns, float* dw, float* db, int N, int C, int J, int64_t HW, b200_stream_t stream);
int b200unet_gen_mul(float* x, int64_t x_ns, const float* mask, int N, int64_t CHW, b200_stream_t stream);
/* ---- attention gates of UNet_attention (Attention_block, Model.py:257-296) on the generic fp32 engine:
 * a = act(scale*y + shift), act: 0 identity (BatchNorm of W_q / W_x), 1 relu, 2 sigmoid (psi) */
int b200unet_gen_bn_act_fwd(const float* y, int64_t y_ns, const float* scale, const float* shift, float* a, int64_t a_ns,
    int N, int C, int HW, int act, b200_stream_t stream);
/* BatchNorm backward with (relu = 1) or without (relu = 0) the ReLU mask; otherwise as b200unet_gen_bn_relu_bwd_*. */
int b200unet_gen_bn_bwd_reduce(const float* g, int64_t g_ns, const float* y, int64_t y_ns, const float* scale,
    const float* shift, const float* mean, const float* rstd, double* sums, int N, int C, int HW, int relu,
    b200_stream_t stream);
int b200unet_gen_bn_bwd_apply(const float* g, int64_t g_ns, const float* y, int64_t y_ns, const float* gamma,
    const float* scale, const float* shift, const float* mean, const float* rstd, const double* sums, double count,
    const double* sums_local, float* dy, int64_t dy_ns, float* dgamma, float* dbeta, int N, int C, int HW, int relu,
    b200_stream_t stream);
/* e = relu(a + b) (Model.py:293) and d = de * [e > 0], dense tensors of `total` elements */
int b200unet_gen_add_relu(const float* a, const float* b, float* e, int64_t total, b200_stream_t stream);
int b200unet_gen_relu_bwd(const float* de, const float* e, float* d, int64_t total, b200_stream_t stream);
/* out[n,c,q] = x[n,c,q] * gate[n,q] (Model.py:295); backward: dx = dout * gate and
 * dpre[n,q] = (sum_c dout*x) * gate*(1-gate) = gradient w.r.t. the input of the sigmoid that produced `gate`. */
int b200unet_gen_gate_fwd(const float* x, int64_t x_ns, const float* gate, float* out, int64_t out_ns, int N, int C,
    int64_t HW, b200_stream_t stream);
int b200unet_gen_gate_bwd(const float* dout, int64_t dout_ns, const float* x, int64_t x_ns, const float* gate, float* dx,
    int64_t dx_ns, float* dpre, int N, int C, int64_t HW, b200_stream_t stream);
/* dst[n,:] += src[n,:] over NCHW views (gradient accumulation where a tensor has two consumers) */
int b200unet_gen_add_inplace(float* dst, int64_t dst_ns, const float* src, int64_t src_ns, int N, int64_t CHW,
    b200_stream_t stream);

/* ---- fused optimizer step (SURVEY.md 8f-1; reference: torch.optim.SGD built in train.py:341-347, stepped in
 * Trainer.py:719-725). torch.optim.SGD arithmetic on the fp32 master parameter (weight decay, momentum, dampening,
 * nesterov; first_step = the momentum buffer is initialised with the gradient) fused with the bf16 re-cast of the
 * two GEMM operands. grad == NULL only refreshes the operands. momentum_buf may be NULL when momentum == 0. */
int b200unet_sgd_conv3x3_weight(float* w_oihw, const float* grad, float* momentum_buf, void* w_fprop, void* w_dgrad,
                                int K, int C, float lr, float momentum, float dampening, float weight_decay,
                                int nesterov, int first_step, b200_stream_t stream);
int b200unet_sgd_convt2x2_weight(float* w, const float* grad, float* momentum_buf, void* w_fprop, void* w_dgrad,
                                 int Cin, int Cup, float lr, float momentum, float dampening, float weight_decay,
                                 int nesterov, int first_step, b200_stream_t stream);
/* the same update for `count` small fp32 tensors (HOST arrays of device pointers / element counts) in one launch
 * per 48 tensors: BatchNorm affine parameters, biases, the 1x1 head, inc.conv1. */
int b200unet_sgd_small(float* const* w, const float* const* grad, float* const* momentum_buf, const int* numel,
                       int count, float lr, float momentum, float dampening, float weight_decay, int nesterov,
                       int first_step, b200_stream_t stream);
/* All conv3x3 weights (kind 0; dim_a = K, dim_b = C) or all ConvTranspose2d weights (kind 1; dim_a = Cin, dim_b = Cup) of a
 * network in ONE launch (HOST arrays of device pointers / dims): most weight tensors are a few tiles, so a launch per tensor
 * is latency-bound. Same arithmetic and operand outputs as the single-tensor entry points above. */
int b200unet_sgd_weights(int kind, float* const* w, const float* const* grad, float* const* momentum_buf,
                         void* const* w_fprop, void* const* w_dgrad, const int* dim_a, const int* dim_b, int count, float lr,
                         float momentum, float dampening, float weight_decay, int nesterov, int first_step,
                         b200_stream_t stream);

/* ---- the same fused pass for Adam (train.py:341-343 `optim.Adam(params, lr, weight_decay)`; configseros.yml:15;
 * Trainer.py:1009): torch.optim.Adam arithmetic - g += weight_decay*w; exp_avg = lerp(exp_avg, g, 1-beta1);
 * exp_avg_sq = beta2*exp_avg_sq + (1-beta2)*g*g; w -= step_size * exp_avg / (sqrt(exp_avg_sq)*inv_sqrt_bc2 + eps) with
 * step_size = lr/(1-beta1^t), inv_sqrt_bc2 = 1/sqrt(1-beta2^t) computed by the host - plus the bf16 GEMM operands.
 * first_step != 0: the moment buffers are uninitialised (treated as zero). */
int b200unet_adam_conv3x3_weight(float* w_oihw, const float* grad, float* exp_avg, float* exp_avg_sq, void* w_fprop,
                                 void* w_dgrad, int K, int C, double beta1, double beta2, float eps, float weight_decay,
                                 float step_size, float inv_sqrt_bc2, int first_step, b200_stream_t stream);
int b200unet_adam_convt2x2_weight(float* w, const float* grad, float* exp_avg, float* exp_avg_sq, void* w_fprop,
                                  void* w_dgrad, int Cin, int Cup, double beta1, double beta2, float eps, float weight_decay,
                                  float step_size, float inv_sqrt_bc2, int first_step, b200_stream_t stream);
int b200unet_adam_small(float* const* w, const float* const* grad, float* const* exp_avg, float* const* exp_avg_sq,
                        const int* numel, int count, double beta1, double beta2, float eps, float weight_decay,
                        float step_size, float inv_sqrt_bc2, int first_step, b200_stream_t stream);
int b200unet_adam_weights(int kind, float* const* w, const float* const* grad, float* const* exp_avg,
                          float* const* exp_avg_sq, void* const* w_fprop, void* const* w_dgrad, const int* dim_a,
                          const int* dim_b, int count, double beta1, double beta2, float eps, float weight_decay,
                          float step_size, float inv_sqrt_bc2, int first_step, b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200UNET_H_ */
