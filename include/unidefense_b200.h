/* libunidefense_b200.so -- C ABI of the B200-native UniDefense dual-space reconstruction path.
 *
 * The reference (VISION-SJTU/UniDefense) is pure Python/PyTorch and has no FFI; its boundary for
 * this path is the nn.Module contract of model/unidefense.py (forward() -> cls_out/rec/loss_dict).
 * Each entry point below replaces the torch call sequence cited next to it; the Python mirror
 * of the reference interface (unidefense_b200/model, /loss) binds these through ctypes.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer into caller-owned memory (torch's caching allocator);
 *    the library never allocates or frees caller tensors.  It owns only immutable per-size
 *    twiddle tables, created lazily, cached for the process lifetime (mutex-guarded).
 *  - tensors are fp32, NCHW, contiguous.  Spectra use the reference's channel-planar
 *    cat([re, im], dim=1) layout ([N, 2C, H, W/2+1]), never interleaved complex.
 *  - `stream` is the CUDA stream to launch on (the shim passes torch's current stream);
 *    entry points are re-entrant and may be called from autograd's worker threads.
 *  - return 0 on success, a negative UD_ERR_* code otherwise; ud_last_error() returns a
 *    thread-local message.  No exceptions cross this boundary.
 *  - workspaces are passed in by the caller; *_workspace_bytes() say how large.
 *  - the first call for a new FFT length / resize pair builds its table with cudaMalloc + a synchronous copy:
 *    warm every shape up once before capturing calls into a CUDA graph (all later calls are capture-safe).
 *  - reductions are fixed-order (bitwise reproducible) except ud_recon_tail_bwd's g_dec and ud_bilinear_ac_bwd,
 *    whose transposed resize accumulates with float atomics.  The input-gradient outputs (g_x of ud_recon_tail_bwd,
 *    ud_attn_prep_bwd, ud_gaussian_blur5_bwd, ud_downscale_nearest_bwd; g_diff of ud_dyfi_mask_bwd) are gathers
 *    written once per element: bitwise reproducible.  ud_attack_step's per-sample norms are fixed-order too.
 *    ud_corrupt writes every output element once from a fixed-order computation: bitwise reproducible.
 */
#ifndef UNIDEFENSE_B200_H
#define UNIDEFENSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if !defined(__CUDA_RUNTIME_H__) && !defined(__DRIVER_TYPES_H__)
typedef struct CUstream_st* cudaStream_t;
#endif

#if defined(__GNUC__)
#define UD_API __attribute__((visibility("default")))
#else
#define UD_API
#endif

#define UD_B200_VERSION 103
#define UD_FFT_MAX_N 1024

#define UD_ACT_NONE 0
#define UD_ACT_RELU 1   /* nn.ReLU            (model/unidefense.py:277,457) */
#define UD_ACT_SWISH 2  /* MemoryEfficientSwish (model/unidefense.py:56; efficientnet/utils.py:66-82) */

UD_API const char* ud_last_error(void);
UD_API int ud_version(void);
/* Kernels launched by this library since load (process-wide, monotonic): bench.py's gpu_launches. */
UD_API long long ud_launch_count(void);
/* 1 when n-point line FFTs run on the mixed-radix plan (prime factors <= 23, n <= UD_FFT_MAX_N);
 * ud_fft_size_any: 1 for every 1 <= n <= UD_FFT_MAX_N (other sizes run Bluestein's algorithm). */
UD_API int ud_fft_size_supported(int n);
UD_API int ud_fft_size_any(int n);

/* ---- a1: reconstruction-loss tail --------------------------------------------------------
 * Replaces model/unidefense.py:244-253 (Eb4), :423-433 (Res18), :618-628 (Res50):
 *   interpolate(dec, x.shape[-2:]) ; abs(rec-x).mean ; rfft2 x2 ; cat ; abs ; tensor_split ; mean.
 * dec [N,C,h,w], x [N,C,H,W] -> rec [N,C,H,W], spatial [N], freq [N].
 * Any 1 <= H, W <= UD_FFT_MAX_N.  The decoder width w shares shared memory with one row FFT: every w <= 2214 fits
 * at every W; a wider decoder that does not fit is rejected (UD_ERR_UNSUPPORTED) before any launch.
 * signs (nullable; ud_recon_tail_signs_bytes) receives 1 byte per spectral bin (sign codes of
 * Re/Im dF) and is what backward needs instead of the two saved spectra.                    */
UD_API size_t ud_recon_tail_workspace_bytes(int N, int C, int h, int w, int H, int W);
UD_API size_t ud_recon_tail_signs_bytes(int N, int C, int H, int W);
UD_API int ud_recon_tail_fwd(const float* dec, const float* x, float* rec, float* spatial, float* freq,
                             uint8_t* signs, void* ws, size_t ws_bytes, int N, int C, int h, int w, int H,
                             int W, int norm_ortho, cudaStream_t stream);
/* g_dec [N,C,h,w] = d(sum_n g_spatial[n]*spatial[n] + g_freq[n]*freq[n]) / d dec
 * (torch autograd of the lines above: abs -> sgn, fft_r2c_backward, upsample_bilinear2d_backward).
 * Samples with g_spatial[n]==g_freq[n]==0 (the engine's fake rows, abstract_engine.py:241,249)
 * cost nothing.
 * g_x [N,C,H,W] is the input-image gradient (x is differentiated in the reference: rec - x at
 * model/unidefense.py:245 and rfft2(x) at :247):
 *   g_x = -(g_spatial[n]*sign(d)/(C*H*W) + fft_r2c_backward(g_freq[n]*sign(dF)/(C*H*Wh)))   (d = rec - x),
 * stored at full resolution by the pass that holds it before the transposed resize; samples with
 * g_spatial[n]==g_freq[n]==0 get g_x = 0.  g_dec and g_x are each nullable (not both).         */
UD_API int ud_recon_tail_bwd(const float* dec, const float* x, const uint8_t* signs, const float* g_spatial,
                             const float* g_freq, float* g_dec, float* g_x, void* ws, size_t ws_bytes, int N, int C,
                             int h, int w, int H, int W, int norm_ortho, cudaStream_t stream);

/* ---- a2: decoder epilogues ------------------------------------------------------------------
 * nn.InstanceNorm2d(C, affine) + MemoryEfficientSwish / nn.ReLU after every decoder conv
 * (model/unidefense.py:61-98, :286-305, :466-497): x [N,C,HW] -> y = act((x-mu)/sqrt(var+eps)*gamma+beta)
 * per (n,c) plane, biased variance, no running stats.  mean/rstd [N*C] are saved for backward.
 * ymean (nullable) [N*C] receives mean_hw(y): the triplet features dec_out.mean([-2,-1])
 * (model/unidefense.py:232-236) for free.  gamma/beta may be NULL (affine=False).              */
UD_API int ud_in_act_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean,
                         float* rstd, float* ymean, int N, int C, int HW, float eps, int act,
                         cudaStream_t stream);
UD_API size_t ud_in_act_bwd_workspace_bytes(int N, int C);
/* gx [N,C,HW], ggamma/gbeta [C] (nullable).  g_ymean (nullable) [N*C] is the gradient w.r.t. ymean.
 * Swish backward follows SwishImplementation.backward (model/efficientnet/utils.py:73-77).       */
UD_API int ud_in_act_bwd(const float* x, const float* gy, const float* gamma, const float* beta,
                         const float* mean, const float* rstd, const float* g_ymean, float* gx, float* ggamma,
                         float* gbeta, void* ws, size_t ws_bytes, int N, int C, int HW, int act,
                         cudaStream_t stream);
/* bf16 in / bf16 out variants (SURVEY §8b "bf16 in/out variants with fp32 accumulation"): x, y, gy, gx are bf16
 * [N,C,HW] (torch.bfloat16 storage, passed as void*); statistics, affine parameters, ymean and all arithmetic stay fp32;
 * stores round to nearest even.  Under bf16 autocast the decoder convolutions emit and consume bf16, so these calls
 * remove the fp32 <-> bf16 casting passes the reference composition makes around every InstanceNorm
 * (bit-identical to cast -> fp32 kernel -> cast).                                                         */
UD_API int ud_in_act_fwd_bf16(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                              float* ymean, int N, int C, int HW, float eps, int act, cudaStream_t stream);
UD_API int ud_in_act_bwd_bf16(const void* x, const void* gy, const float* gamma, const float* beta, const float* mean,
                              const float* rstd, const float* g_ymean, void* gx, float* ggamma, float* gbeta, void* ws,
                              size_t ws_bytes, int N, int C, int HW, int act, cudaStream_t stream);
/* nn.Tanh decoder output (model/unidefense.py:101, :307, :499). */
UD_API int ud_tanh_fwd(const float* x, float* y, long long n, cudaStream_t stream);
UD_API int ud_tanh_bwd(const float* y, const float* gy, float* gx, long long n, cudaStream_t stream);

/* ---- a4 / a7: attention() glue -----------------------------------------------------------------
 * F.interpolate(mode='bilinear', align_corners=True) (model/unidefense.py:16) on [planes,h,w] -> [planes,H,W]
 * and its transpose (upsample_bilinear2d_backward; gx is zeroed by the call).                       */
UD_API int ud_bilinear_ac_fwd(const float* x, float* y, int planes, int h, int w, int H, int W, cudaStream_t stream);
UD_API int ud_bilinear_ac_bwd(const float* gy, float* gx, int planes, int h, int w, int H, int W,
                              cudaStream_t stream);
/* Error maps (model/unidefense.py:126-134,:148; no grad): pred [N,C,hp,wp] and x [N,C,Hx,Wx] are resized
 * to (h,w); spat_diff [N,C,h,w] = |p-xs|; freq_diff [N,2C,h,w/2+1] = |cat(re,im) rfft2(p-xs)|.      */
UD_API int ud_attn_prep(const float* pred, const float* x, float* spat_diff, float* freq_diff, int N, int C, int hp,
                        int wp, int Hx, int Wx, int h, int w, int norm_ortho, cudaStream_t stream);
/* Its gradient w.r.t. x (model/unidefense.py:127-134: x is resized and enters p - xs; pred is detached by the caller,
 * :213/:393/:586): d = down(pred) - down(x) is recomputed at (h,w),
 *   g_d = sign(d)*g_spat_diff + fft_r2c_backward(sign(cat(re,im) rfft2(d)) * g_freq_diff),
 *   g_x [N,C,Hx,Wx] = -(transposed align-corners resize)(g_d), evaluated as a gather (no atomics, fully written).
 * g_spat_diff [N,C,h,w] and g_freq_diff [N,2C,h,w/2+1] are each nullable.  Same shapes as ud_attn_prep; N*C <= 65535. */
UD_API int ud_attn_prep_bwd(const float* pred, const float* x, const float* g_spat_diff, const float* g_freq_diff,
                            float* g_x, int N, int C, int hp, int wp, int Hx, int Wx, int h, int w, int norm_ortho,
                            cudaStream_t stream);
/* ud_rfft2: torch.fft.rfft2 + cat([re,im],1) (model/unidefense.py:135-136): x [N,C,h,w] -> xf [N,2C,h,w/2+1].
 * adjoint_of_inverse=1 gives irfft2's backward (fft_c2r_backward: interior columns doubled, inverse normalisation;
 * SURVEY App. B.3).
 * ud_irfft2: torch.complex(*tensor_split(xf,2,1)) + irfft2(s=(h,w)) (model/unidefense.py:142-145): xf [N,2C,h,w/2+1]
 * (optionally multiplied on load by mask [N,h*(w/2+1)]) -> y [N,C,h,w].  adjoint_of_forward=1 gives rfft2's backward
 * (fft_r2c_backward: zero-padded half spectrum, no mirroring; SURVEY App. B.2).
 * Both take ANY 1 <= h, w <= UD_FFT_MAX_N (torch.fft.rfft2 / irfft2 as also called at model/unidefense.py:246-249,
 * model/modules.py:43-54, model/efficientnet/exp.py:55-65, model/resnet/exp.py:44-54): mixed radix when every prime
 * factor is <= 23, Bluestein otherwise.  Planes with h, w <= 64 take the workspace-free small-plane path; larger planes
 * need ws of ud_rfft2_workspace_bytes() (the row-transformed half spectrum, [N*C][h][w/2+1] complex).             */
UD_API size_t ud_rfft2_workspace_bytes(int N, int C, int h, int w);
UD_API int ud_rfft2(const float* x, float* xf, void* ws, size_t ws_bytes, int N, int C, int h, int w, int norm_ortho,
                    int adjoint_of_inverse, cudaStream_t stream);
UD_API int ud_irfft2(const float* xf, const float* mask, float* y, void* ws, size_t ws_bytes, int N, int C, int h,
                     int w, int norm_ortho, int adjoint_of_forward, cudaStream_t stream);
/* out = (1-s)*smask*emb + s*ff + res, s = sigmoid(*fuse_coef) (model/unidefense.py:153-155).
 * emb, ff, res, out [N,C,HW]; smask [N,HW]; res = dropout(emb.clone()) or NULL (= emb).             */
UD_API int ud_attn_fuse_fwd(const float* emb, const float* smask, const float* ff, const float* res,
                            const float* fuse_coef, float* out, int N, int C, int HW, cudaStream_t stream);
UD_API size_t ud_attn_fuse_bwd_workspace_bytes(int N, int HW);
UD_API int ud_attn_fuse_bwd(const float* emb, const float* smask, const float* ff, const float* g,
                            const float* fuse_coef, float* g_emb, float* g_ff, float* g_smask, float* g_coef,
                            void* ws, size_t ws_bytes, int N, int C, int HW, int res_is_emb, cudaStream_t stream);

/* ---- a5 / a6: dynamic filters (model/modules.py:79-134) ---------------------------------------------
 * Local BatchNorm statistics of x [N,C,HW]: mean[c], m2[c] = sum (x-mean)^2 over N*HW (the caller merges
 * ranks for SyncBatchNorm, engine/forgery_engine.py:142, and derives rstd / running stats).          */
UD_API int ud_bn_stats(const float* x, float* mean, float* m2, int N, int C, int HW, cudaStream_t stream);
UD_API int ud_bn_bwd_reduce(const float* dz, const float* x, const float* mean, const float* rstd, float* sum_dz,
                            float* sum_dz_xh, int N, int C, int HW, cudaStream_t stream);
/* inv_count = 1/(global N*HW) in training, 0 in eval (running stats: pure scaling).                  */
UD_API int ud_bn_bwd_apply(const float* dz, const float* x, const float* mean, const float* rstd,
                           const float* gamma, const float* sum_dz, const float* sum_dz_xh, float inv_count,
                           float* gx, int N, int C, int HW, cudaStream_t stream);
/* The dense projection itself -- FrequencyDynamicFilter.layer1[0] = nn.Conv2d(2C,2C,1) (model/modules.py:82-85),
 * SpatialDynamicFilter.layer1[0] = nn.Conv2d(C,C,3,1,1) (model/modules.py:111-114), bias-free -- as ONE implicit
 * GEMM on the 5th-generation tensor cores (TMA -> 128B-swizzled smem -> tcgen05.mma.kind::tf32 -> TMEM), with the
 * BatchNorm2d batch statistics of layer1[1] produced per M tile in the epilogue.
 *   x_hi [N,H,W,Cin] channels-last fp32 activations, w_hi [Cout, ksize*ksize, Cin] (tap = ky*ksize+kx);
 *   x_lo / w_lo: nullable low parts for "3xTF32" (hi = TF32-rounded value, lo = x - hi): fp32-grade accuracy;
 *   with both NULL the product is plain TF32 (what cuDNN computes under torch's default allow_tf32=True).
 *   y [N,Cout,H,W] (NCHW); part_mean/part_m2 [m_tiles, Cout] and part_cnt [m_tiles] (all three or none):
 *   per-tile mean, sum (x-mean)^2 and pixel count, merged by ud_bn_merge_partials into ud_bn_stats' outputs.
 * Cin % 4 == 0, Cin >= 32, W <= 128.  ud_proj_prep_x / _w build the operand layouts (transpose + split).   */
UD_API int ud_proj_m_tiles(int N, int H, int W, int ksize);
UD_API int ud_proj_prep_x(const float* x_nchw, float* hi, float* lo, int N, int C, int P, cudaStream_t stream);
UD_API int ud_proj_prep_w(const float* w, float* hi, float* lo, int Cout, int Cin, int taps, cudaStream_t stream);
UD_API int ud_proj_fwd(const float* x_hi, const float* x_lo, const float* w_hi, const float* w_lo, float* y,
                       float* part_mean, float* part_m2, float* part_cnt, int N, int H, int W, int Cin, int Cout,
                       int ksize, cudaStream_t stream);
/* Backward of the projections on the same tensor-core kernel:
 *   data gradient   dX = conv(dY, flip(W)^T): ud_proj_fwd with x = dY (channels-last) and the weights re-laid by
 *                   ud_proj_prep_wt ([Cout,Cin,k,k] -> [Cin, k*k flipped, Cout]); output lands NCHW like the forward.
 *   weight gradient (1x1) dW[co,ci] = sum_{n,p} dY[n,co,p] X[n,ci,p]: ud_proj_wgrad_1x1, both operands NCHW [N,C,P],
 *                   K = (sample, 32-pixel chunk) via 3-D TMA boxes; P % 4 == 0.  (The 3x3 weight gradient stays on
 *                   the library: its K blocks are not 128-byte rows for 12x12 / 24x24 planes.)
 *   ud_proj_split: elementwise hi/lo split of an operand for 3xTF32.                                              */
UD_API int ud_proj_prep_wt(const float* w, float* hi, float* lo, int Cout, int Cin, int taps, cudaStream_t stream);
UD_API int ud_proj_split(const float* x, float* hi, float* lo, long long total, cudaStream_t stream);
UD_API int ud_proj_wgrad_1x1(const float* x_hi, const float* x_lo, const float* dy_hi, const float* dy_lo, float* dw,
                             int N, int P, int Cin, int Cout, cudaStream_t stream);
UD_API int ud_bn_merge_partials(const float* part_mean, const float* part_m2, const float* part_cnt, float* mean,
                                float* m2, int tiles, int C, cudaStream_t stream);
/* Everything after layer1's conv: BN-apply + act + channel mean/max + cat(diff) + conv1x1 (w2 [2+D]) +
 * sigmoid -> mask [N,HW]; out [N,Cx,HW] = mask*x (nullable).  proj [N,Cp,HW] is the raw conv output.
 * pmean/pmax [N,HW] and argmax [N,HW] (first index on ties, like torch.max) are saved for backward.   */
UD_API int ud_dyfi_mask_fwd(const float* proj, const float* bn_mean, const float* bn_rstd, const float* gamma,
                            const float* beta, const float* diff, const float* w2, const float* x, float* mask,
                            float* out, float* pmean, float* pmax, int* argmax, int N, int Cp, int D, int Cx, int HW,
                            int act, cudaStream_t stream);
UD_API size_t ud_dyfi_mask_bwd_workspace_bytes(int N, int HW);
/* g_mask [N,HW] / g_out [N,Cx,HW] (either nullable) -> g_x = mask*g_out, dz [N,Cp,HW] (gradient w.r.t.
 * the BN output, to be finished by ud_bn_bwd_*), g_w2 [2+D], and g_diff [N,D,HW] (nullable) = w2[2+k] * d loss / d logit:
 * the gradient of the guide channels cat'ed into layer2's input (model/modules.py:101-103, :130-132), through which the
 * error maps carry x's gradient.                                                                                   */
UD_API int ud_dyfi_mask_bwd(const float* proj, const float* bn_mean, const float* bn_rstd, const float* gamma,
                            const float* beta, const float* diff, const float* w2, const float* x, const float* mask,
                            const float* pmean, const float* pmax, const int* argmax, const float* g_mask,
                            const float* g_out, float* g_x, float* dz, float* g_w2, float* g_diff, void* ws,
                            size_t ws_bytes, int N, int Cp, int D, int Cx, int HW, int act, cudaStream_t stream);

/* ---- a9-a11: losses; each also returns d loss / d input for upstream gradient 1 ------------------
 * AsymmetricalWeightedTripletLoss.forward (loss/triplet_loss.py:75-82): feat [N,c], labels int64 [N]
 * (label-0 rows are the anchors and come first), N <= 128.  gfeat nullable.                         */
UD_API int ud_triplet_fwd(const float* feat, const long long* labels, float* loss, float* gfeat, int N, int c,
                          cudaStream_t stream);
/* FactorizationLoss.forward (loss/calib_loss.py:17-28): emb_a (grad), emb_b [N,F], 2 <= N <= 128.    */
UD_API size_t ud_factorization_workspace_bytes(int N, int F);
UD_API int ud_factorization_fwd(const float* emb_a, const float* emb_b, float* loss, float* g_a, void* ws,
                                size_t ws_bytes, int N, int F, float off_diag_weight, float eps, cudaStream_t stream);
/* KLDivLoss(batchmean, log_target)(log_softmax(pred.flat), log_softmax(gt.flat))
 * (engine/abstract_engine.py:333-346): pred, gt [N,M].                                              */
UD_API size_t ud_mask_kl_workspace_bytes(int N);
UD_API int ud_mask_kl_fwd(const float* pred, const float* gt, float* loss, float* g_pred, void* ws, size_t ws_bytes,
                          int N, int M, cudaStream_t stream);

/* nn.KLDivLoss(reduction="batchmean", log_target=True) (loss/__init__.py:17) with the engine's call
 * signature: both arguments are log-probabilities [N,M] (workspace: ud_mask_kl_workspace_bytes).  */
UD_API int ud_kl_div_log_target_fwd(const float* log_pred, const float* log_target, float* loss, float* g_pred,
                                    void* ws, size_t ws_bytes, int N, int M, cudaStream_t stream);

/* ---- a12: classification loss (engine/abstract_engine.py:256-259, :325-328) ------------------------------------
 * nn.CrossEntropyLoss() on logits [N,K] / int64 targets [N] (mean reduction), and the num_classes == 1 branch
 * nn.BCEWithLogitsLoss() on logits [N] / float targets [N].  g_logits (nullable) = d loss / d logits.            */
UD_API int ud_cross_entropy_fwd(const float* logits, const long long* target, float* loss, float* g_logits, int N,
                                int K, cudaStream_t stream);
UD_API int ud_bce_with_logits_fwd(const float* logits, const float* target, float* loss, float* g_logits, int N,
                                  cudaStream_t stream);

/* ---- a13: FrequencyStyleTransfer (model/modules.py:35-55; no grad) --------------------------------------
 * out = irfft2((lmda*|Fa| + (1-lmda)*|Fb|) * exp(1j*angle(Fa))), Fa/Fb = rfft2 of content/style, ortho;
 * content, style, out [N,C,H,W]; lmda [N] (the reference draws it on the CPU in [0.5, 1)).              */
UD_API size_t ud_freq_style_workspace_bytes(int N, int C, int H, int W);
UD_API int ud_freq_style_transfer(const float* content, const float* style, const float* lmda, float* out, void* ws,
                                  size_t ws_bytes, int N, int C, int H, int W, cudaStream_t stream);

/* a14 -- SpatialStyleTransfer (model/modules.py:59-76; no grad): exact rank matching per (n,c) plane,
 *   out = content + (1-lmda[n]) * style_sorted[rank(content)] - (1-lmda[n]) * content
 * content, style, out [N,C,HW]; lmda [N].  One stable radix sort per plane (style: keys only; content: keys + pixel
 * index with the blend fused into the last pass) through ws of ud_spatial_style_workspace_bytes().  Replaces the
 * reference's two torch.sort + argsort + gather.  Ties keep pixel order (torch.sort leaves it unspecified).   */
UD_API size_t ud_spatial_style_workspace_bytes(int N, int C, int HW);
UD_API int ud_spatial_style_transfer(const float* content, const float* style, const float* lmda, float* out, void* ws,
                                     size_t ws_bytes, int N, int C, int HW, cudaStream_t stream);
/* ---- a15: coral colour-statistics transfer (utils/operation.py:15-45; model/unidefense.py:189-191; no grad) ---------
 * source[n] takes the per-channel mean / unbiased std and the 3x3 "f f^T + I" colour structure of target[n]:
 *   out = sqrt~(cov_t) inv(sqrt~(cov_s)) (s - mean_s)/std_s * std_t + mean_t,  sqrt~(M) = U sqrt(D) Vh^T (the
 *   reference's quirk: Vh transposed again).  The quirk depends on the sign of each singular vector, which the SVD
 *   leaves open (LAPACK and cuSOLVER disagree): this kernel signs every eigenvector so that its largest-magnitude
 *   component is positive; parity with the reference holds modulo that gauge (tests/test_perturb_gpu.py).
 * source, target, out [N,3,HW] fp32; three launches for the whole batch, no host synchronisation.               */
UD_API size_t ud_coral_workspace_bytes(int N, int HW);
UD_API int ud_coral(const float* source, const float* target, float* out, void* ws, size_t ws_bytes, int N, int HW,
                    cudaStream_t stream);

/* ---- a16: stencil / resampling perturbations ---------------------------------------------------------
 * random_blur (model/modules.py:15-16): torchvision gaussian_blur 5x5, sigma 1.1, reflect padding.   */
UD_API int ud_gaussian_blur5(const float* x, float* y, int planes, int H, int W, cudaStream_t stream);
/* downscale (model/modules.py:19-21): nearest by `bottleneck_scale`, then nearest back to HxW.       */
UD_API int ud_downscale_nearest(const float* x, float* y, int planes, int H, int W, float bottleneck_scale,
                                cudaStream_t stream);
/* Their adjoints (torch autograd of model/modules.py:16 and :20-21; pass 2 of training applies them to x):
 * gx [planes,H,W] from gy [planes,H,W].  Blur: the reflected border taps fold back onto the border pixels;
 * downscale: each input pixel sums the gradient of its nearest-index preimage (H + W + 2 ints of shared memory). */
UD_API int ud_gaussian_blur5_bwd(const float* gy, float* gx, int planes, int H, int W, cudaStream_t stream);
UD_API int ud_downscale_nearest_bwd(const float* gy, float* gx, int planes, int H, int W, float bottleneck_scale,
                                    cudaStream_t stream);

/* ---- a17 (next row, first step): glue of the SFConv frequency branch ----------------------------------
 * (model/efficientnet/exp.py:55-65, model/resnet/exp.py:44-54).  spec: interleaved complex64 [N,C,P]
 * (P = h*(w/2+1), torch.fft.rfft2's output); planar: cat([re, im], 1) as [N,2C,P], fp32 or bf16 (bf16=1),
 * NCHW or channels-last [N,P,2C] (nhwc=1, C even).  pack and unpack are each other's autograd adjoint.      */
UD_API int ud_sf_pack(const void* spec, void* planar, int N, int C, int P, int nhwc, int bf16, cudaStream_t stream);
UD_API int ud_sf_unpack(const void* planar, void* spec, int N, int C, int P, int nhwc, int bf16, cudaStream_t stream);
/* out = (1-s)*spat + s*freq, s = sigmoid(*coef) (exp.py:64-65 / :53-54).  spat, out (and their gradients):
 * dtype/layout per (bf16, nhwc); freq, g_freq: fp32 NCHW [N,C,P].                                           */
UD_API int ud_sf_mix_fwd(const void* spat, const float* freq, const float* coef, void* out, int N, int C, int P,
                         int nhwc, int bf16, cudaStream_t stream);
UD_API size_t ud_sf_mix_bwd_workspace_bytes(int N, int C, int P);
UD_API int ud_sf_mix_bwd(const void* g_out, const void* spat, const float* freq, const float* coef, void* g_spat,
                         float* g_freq, float* g_coef, void* ws, size_t ws_bytes, int N, int C, int P, int nhwc,
                         int bf16, cudaStream_t stream);

/* ---- a19: projected-gradient attack step (PGD / FGSM robustness evaluation) ---------------------------------------
 * One iteration's image-sized work for a batch, per sample n, mirroring oracle/attack.py operation for operation in
 * fp32 with explicit rounding (no FMA contraction; sign(0) = 0 as torch.sign):
 *  1. select: if loss[n] > best_loss[n] (strict: a NaN loss never improves), best_loss[n] = loss[n] and
 *     x_best[n] = x_adv[n] as it was BEFORE this call's step; other samples keep x_best / best_loss bit for bit.
 *  2. step (skipped when g == NULL: "select only", for the iterate after the last forward):
 *     UD_NORM_LINF: x_adv = clamp(x0 + clamp((x_adv + alpha*sign(g)) - x0, -eps, eps), lo, hi)
 *     UD_NORM_L2:   u = g / (||g_n||_2 + 1e-12); d = x_adv + alpha*u - x0; d *= min(1, eps/||d_n||_2) (0/0 -> 1);
 *                   x_adv = clamp(x0 + d, lo, hi)
 * x0, x_adv, g, x_best [N, per_sample] (any per_sample >= 1); loss, best_loss, eps, alpha [N], all fp32 device memory
 * (eps / alpha on the device so one captured graph serves an eps sweep; both may be NULL for a select-only call).
 * x_adv, best_loss, x_best are updated in place; x_best must not alias x_adv.  The L2 norms are fixed-order sums of
 * per-CTA partials kept in ws (ud_attack_workspace_bytes): two calls on the same inputs are bitwise identical.
 * Launches: 2 (L-inf, select only) or 3 (L2).  N <= 65535.                                                         */
#define UD_NORM_LINF 0
#define UD_NORM_L2 2
UD_API size_t ud_attack_workspace_bytes(int N, long long per_sample);
UD_API int ud_attack_step(const float* x0, float* x_adv, const float* g, const float* loss, float* best_loss,
                          float* x_best, const float* eps, const float* alpha, float lo, float hi, int norm, int N,
                          long long per_sample, void* ws, size_t ws_bytes, cudaStream_t stream);

/* ---- a20: image corruptions (corruption-robustness evaluation; DeeperForensics-1.0 / LipForensics protocol) -----------
 * y = corruption of x, x and y fp32 [N, 3, H, W] (channels R, G, B, values in [lo, hi]; y must not overlap x).  Each
 * kind maps x to 8-bit levels p = clamp(rint((x - lo)*s), 0, 255) with s = 255/(hi - lo) (fp64 on the host, used as
 * fp32), corrupts p, rounds with rint, clamps to [0, 255] and writes y = lo + p'*(1/s): outputs lie on the 8-bit grid.
 * Colour space: JFIF full-range BT.601 on levels, Y = .299R + .587G + .114B, Cb = -.168736R - .331264G + .5B + 128,
 * Cr = .5R - .418688G - .081312B + 128; inverse R = Y + 1.402(Cr-128), G = Y - .344136(Cb-128) - .714136(Cr-128),
 * B = Y + 1.772(Cb-128).  `param` is the severity parameter:
 *  SATURATION s in [0, 1]: Cb' = 128 + (Cb-128)*s, likewise Cr, back to RGB.
 *  CONTRAST   c in [0, 1]: p' = p*c.
 *  BLOCK      k in 0..4096: k 8x8 squares set to level 128 in all channels; square j's top-left corner is
 *             r = (u0*(H-7)) >> 32, c = (u1*(W-7)) >> 32 (64-bit products) with (u0, u1, ...) = Philox4x32-10(ctr =
 *             (j, id_lo, id_hi, 0), key = (seed_lo, seed_hi ^ 0x424C4F43)).  H, W >= 8.
 *  NOISE      sigma^2 in [0, 1]: in YCbCr/255 add sigma*z to Y, Cb, Cr; z0, z1 by Box-Muller from words (a, b) and z2 from
 *             (c, d) of Philox4x32-10(ctr = (h*W + w, id_lo, id_hi, 0), key = (seed_lo, seed_hi ^ 0x4E4F4953)), with
 *             u1 = (a + 0.5)*2^-32, u2 = b*2^-32, z0 = sqrt(-2 ln u1) cos(2 pi u2), z1 = ... sin(2 pi u2).
 *  BLUR       odd k in 1..31: separable Gaussian, w_i ~ exp(-i^2 / (2 sigma^2)), sigma = k/6, normalised, |i| <= (k-1)/2;
 *             reflect-101 borders (OpenCV's default).  H, W > (k-1)/2.
 *  PIXELATE   f in 1..64: mean of each f x f cell (partial cells at the bottom / right average their valid pixels),
 *             rounded, replicated over the cell.
 *  JPEG       q in 1..100: baseline JPEG round trip, 4:2:0: YCbCr; chroma 2x2 mean (edge replication at odd sizes);
 *             planes padded to whole 8x8 blocks by edge replication; per block orthonormal DCT-II of v - 128 (JPEG's
 *             FDCT scaling), quantised rha(F/Q)*Q (rha: round half away from zero) with the ITU-T T.81 Annex K tables
 *             scaled as libjpeg does (S = 5000/q if q < 50 else 200 - 2q; Q = clamp((T*S + 50) div 100, 1, 255)),
 *             orthonormal IDCT + 128; chroma upsampled with libjpeg's triangle ("fancy") filter; back to RGB.
 *             ws = ud_corrupt_workspace_bytes(JPEG, N, H, W) bytes (0 for every other kind).
 * ids: int64 [N] device array keying the random kinds per sample (id_lo / id_hi its two 32-bit halves), or NULL for
 * ids 0..N-1, so image i gets the same corruption in any batch.  saturation, contrast, block and pixelate are
 * bit-identical to oracle/corrupt.py (fp32, explicit rounding); noise, blur and jpeg restate its fp64 definitions in
 * fp32 (jpeg's forward DCT and quantisation in fp64).  Launches: 1, or 2 for block and jpeg.  N <= 65535, H, W <= 8192. */
#define UD_CORRUPT_SATURATION 0
#define UD_CORRUPT_CONTRAST 1
#define UD_CORRUPT_BLOCK 2
#define UD_CORRUPT_NOISE 3
#define UD_CORRUPT_BLUR 4
#define UD_CORRUPT_PIXELATE 5
#define UD_CORRUPT_JPEG 6
UD_API size_t ud_corrupt_workspace_bytes(int kind, int N, int H, int W);
UD_API int ud_corrupt(const float* x, float* y, const long long* ids, int N, int H, int W, int kind, float param,
                      unsigned long long seed, float lo, float hi, void* ws, size_t ws_bytes, cudaStream_t stream);

/* ---- §8(e): the exchange step -- SyncBatchNorm statistics over NVLink peer memory ----------------------------------
 * Replaces the two per-layer collectives of torch.nn.SyncBatchNorm (engine/forgery_engine.py:142 converts all 99
 * BatchNorms of UDEB4): all_gather of [mean, invstd|M2, count] forward, all_reduce of [sum dy, sum dy*xmu] backward.
 * Every rank owns one buffer (ud_comm_alloc: cudaMalloc + CUDA IPC handle, 64 bytes) that all ranks of the box map
 * (ud_comm_open); ud_comm_gather is ONE single-CTA kernel per rank: remote stores of my vector into every rank's
 * buffer, release-flag, acquire-spin on my own buffer, local copy (reduce=0: dst [world,count]) or fixed-order sum
 * (reduce=1: dst [count]).  Plain kernel launches: CUDA-graph capturable, no host synchronisation, no NCCL.
 * All ranks must issue the same sequence of gathers.  count <= max_count given at creation; world <= 16.          */
UD_API size_t ud_comm_buffer_bytes(int world, int max_count);
UD_API int ud_comm_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_out);
UD_API int ud_comm_open(const void* ipc_handle, void** peer_ptr);
UD_API int ud_comm_create(void* const* peers, int rank, int world, int max_count, void** comm_out);
UD_API int ud_comm_gather(void* comm, const float* src, float* dst, int count, int reduce, cudaStream_t stream);
UD_API int ud_comm_error(void* comm);

#ifdef __cplusplus
}
#endif
#endif /* UNIDEFENSE_B200_H */
