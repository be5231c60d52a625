/* C-ABI of libunetsulc_b200.so — the B200-native (sm_100a) hot path behind UnetPatternSulciLabelling.
 *
 * Everything here replaces arithmetic that the reference reaches through the `deepsulci` import boundary
 * (reference pattern_class.py:19-23): `UNet3D.forward/backward` (training.py:206-211), `nn.CrossEntropyLoss`
 * + `torch.max` on its output (training.py:207-208), `optim.SGD.step` (training.py:212), the Softmax scores
 * gathered by `labeling()` (pattern_class.py:266-277), `cutting(...)` (pattern_class.py:230) and the counters
 * behind `esi_score(...)` (training.py:223-225).  The Python host side (2022_pauriau_unetsulc_b200/ops.py) binds
 * these with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; all pointers are DEVICE pointers unless stated otherwise
 *   - activations: NDHWC bf16, addressed as base[(voxel) * ld + coff + c] ("channel window" of a wider buffer)
 *   - every function returns 0 on success, <0 on error; b2_last_error() returns the thread-local message
 *   - re-entrant; work is enqueued on the cudaStream_t passed in; no allocation, no host synchronisation
 *   - the caller owns every buffer, including workspaces (sizes from the *_workspace_bytes queries)
 *   - no CPU fallback: unsupported shapes are hard errors
 */
#ifndef UNETSULC_B200_H_
#define UNETSULC_B200_H_

#include <cuda_runtime_api.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* b2_last_error(void);

/* ---- 3x3x3 stride-1 pad-1 Conv3d (the 14 convs inside deepsulci UNet3D; training.py:206, 211) -------------------
 * Implicit GEMM on tcgen05/TMEM fed by TMA.  fprop: x = layer input, wpack = fprop pack, relu=1.
 * dgrad: x = dY, wpack = dgrad pack, Cin/Cout swapped, relu=0.  y_is_fp32 selects a fp32 output buffer.
 * Cin and Cout: multiples of 16 (K chunks of 64, 32 or 16 channels; N tiles of up to 256 channels).               */
int b2_conv3d_igemm(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff,
                    int y_is_fp32, int N, int D, int H, int W, int Cin, int Cout, int relu, cudaStream_t stream);

/* b2_conv3d_igemm with an fp32 workspace: layers with fewer output tiles than half the SMs (12x14x12 level) are split
 * over the 27 taps (split-K) into the workspace and reduced (+ReLU, bf16) by a second kernel.                      */
long long b2_conv3d_splitk_workspace_bytes(int N, int D, int H, int W, int Cout);
int b2_conv3d_igemm_splitk(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff, int N,
                           int D, int H, int W, int Cin, int Cout, int relu, void* workspace,
                           long long workspace_bytes, cudaStream_t stream);

/* ---- statistics accumulators ------------------------------------------------------------------------------------
 * GroupNorm statistics travel between kernels as order-independent fixed-point accumulators: int64 [C][4] per layer =
 * {sum_hi, sum_lo, sq_hi, sq_lo} (integer part + fraction in units of 2^-32: every fp32 contribution is represented
 * to within 2^-33, exactly when its magnitude is >= 2^-9), filled with integer atomics by the
 * kernel that PRODUCES the tensor and turned into mean / rstd / coefficients by a one-block finalize: no per-block
 * partial buffers, no statistics pass over the tensor, bit-identical run to run.  The caller zeroes the accumulators before the producer runs.
 *
 * fprop with the statistics of the stored (bf16, post-ReLU) output fused into the epilogue (batch 1, Cout <= 256). */
int b2_conv3d_igemm_stats(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff, int N,
                          int D, int H, int W, int Cin, int Cout, int relu, long long* stat_acc, cudaStream_t stream);
/* dgrad with the GroupNorm-BACKWARD statistics (sum dX, sum dX*r per channel) of the producing layer fused into the
 * epilogue; r = that layer's stored relu(conv), dense bf16 [V][Cout]; dX is written densely (ld = Cout).            */
int b2_conv3d_igemm_bstats(const void* x, int ldx, int x_coff, const void* wpack, void* y, int N, int D, int H, int W,
                           int Cin, int Cout, const void* r, long long* stat_acc, cudaStream_t stream);
/* accumulators -> mean_rstd fp32 [C][2] + scale_shift fp32 [C][2] (one small block; then b2_relu_gn_apply), and the
 * backward counterpart: accumulators of (sum dy, sum dy*r) -> coefficients, dgamma, dbeta (may be NULL) + the apply
 * pass, without a statistics pass over (dy, r).  Batch 1.  workspace >= C*16 bytes.                                 */
int b2_relu_gn_finalize_acc(const long long* stat_acc, long long V, int C, int G, float eps, const float* gamma,
                            const float* beta, float* mean_rstd, float* scale_shift, cudaStream_t stream);
int b2_relu_gn_bwd_acc(const long long* stat_acc, const void* dy, int lddy, int dy_coff, const void* r, long long V,
                       int C, int G, const float* gamma, const float* mean_rstd, void* dr, float* dgamma,
                       float* dbeta, void* workspace, long long workspace_bytes, const long long* dy_row_labels,
                       cudaStream_t stream);   /* dy_row_labels (may be NULL): see b2_head_ce_bstats */

/* dW[co][ci][3][3][3] (fp32, PyTorch layout) = sum_v dY[v,co] * X[v+off,ci].  Cin: 16 or a multiple of 32; Cout: a
 * multiple of 32.  The workspace query returns -1 for any other shape.                                             */
long long b2_conv3d_wgrad_workspace_bytes(int N, int D, int H, int W, int Cin, int Cout);
int b2_conv3d_wgrad(const void* x, int ldx, int x_coff, const void* dy, int ldy, int y_coff, float* dw,
                    void* workspace, long long workspace_bytes, int N, int D, int H, int W, int Cin, int Cout,
                    cudaStream_t stream);

/* The same in two halves, so that the split reductions of SEVERAL layers run as one launch (13 short latency-bound
 * launches per step otherwise): b2_conv3d_wgrad_partial runs the tensor-core kernel and leaves the split partials in
 * `workspace` (private to that layer until reduced; *splits_out / *swapped_out describe their layout);
 * b2_wgrad_reduce_multi reduces `count` layers (HOST arrays of `count` entries) into their dW tensors.            */
int b2_conv3d_wgrad_partial(const void* x, int ldx, int x_coff, const void* dy, int ldy, int y_coff, void* workspace,
                            long long workspace_bytes, int N, int D, int H, int W, int Cin, int Cout,
                            int* splits_out, int* swapped_out, cudaStream_t stream);
int b2_wgrad_reduce_multi(const float* const* ws, float* const* dw, const int* splits, const int* cin,
                          const int* cout, const int* swapped, int count, cudaStream_t stream);

/* encoders.0.conv1 (Cin = 1): direct convolution on the fp32 [N,D,H,W] skeleton volume (dataset.py:78-80).
 * Cout = 16, 32 or 64 (init_channel_number 32 or 64).                                                              */
int b2_conv3d_first_fwd(const float* x, const float* w, void* y, int ldy, int y_coff, int N, int D, int H, int W,
                        int Cout, int relu, cudaStream_t stream);
/* same, with the GroupNorm statistics of the stored output fused in (batch 1): stat_acc int64 [Cout][4], see above  */
int b2_conv3d_first_fwd_stats(const float* x, const float* w, void* y, int ldy, int y_coff, int N, int D, int H, int W,
                              int Cout, int relu, long long* stat_acc, cudaStream_t stream);
long long b2_conv3d_first_wgrad_workspace_bytes(int Cout);
int b2_conv3d_first_wgrad(const float* x, const void* dy, int lddy, int dy_coff, float* dw, void* workspace,
                          long long workspace_bytes, int N, int D, int H, int W, int Cout, cudaStream_t stream);

/* ---- ReLU + GroupNorm ('crg' order), r = relu(conv) is produced by the conv epilogue ---------------------------
 * counters: device int32 [N+1], zero before the first call; the kernels leave it zero ("last block done" tickets). */
long long b2_gn_workspace_bytes(int N, int C);
int b2_relu_gn_stats(const void* r, int N, long long V, int C, int G, float eps, const float* gamma,
                     const float* beta, float* mean_rstd, float* scale_shift, void* workspace,
                     long long workspace_bytes, int* counters, cudaStream_t stream);
/* y = GN(r); pooled != NULL additionally writes MaxPool3d(2,2,0)(y) in the same pass (encoder -> next level)      */
int b2_relu_gn_apply(const void* r, int N, int D, int H, int W, int C, const float* scale_shift, void* y, int ldy,
                     int y_coff, void* pooled, cudaStream_t stream);
long long b2_relu_gn_bwd_workspace_bytes(int N, int C);
int b2_relu_gn_bwd(const void* dy, int lddy, int dy_coff, const void* r, int N, long long V, int C, int G,
                   const float* gamma, const float* mean_rstd, void* dr, float* dgamma, float* dbeta,
                   void* workspace, long long workspace_bytes, int* counters, cudaStream_t stream);

/* ---- MaxPool3d(2) backward (+ skip gradient add), trilinear upsample + concat and its backward ------------------ */
int b2_maxpool3d_bwd_add(const void* y, int ldy, int y_coff, const void* dskip, int ldd, int d_coff,
                         const void* dpool, void* out, int N, int D, int H, int W, int C, cudaStream_t stream);
/* same (batch 1) + the GroupNorm-backward statistics (sum out, sum out*r) of the layer whose output gradient `out` is,
 * accumulated into stat_acc int64 [C][4]; r = that layer's saved relu(conv), dense bf16 [V][C]                      */
int b2_maxpool3d_bwd_add_bstats(const void* y, int ldy, int y_coff, const void* dskip, int ldd, int d_coff,
                                const void* dpool, void* out, int N, int D, int H, int W, int C, const void* r,
                                long long* stat_acc, cudaStream_t stream);
int b2_upcat_fwd(const void* x, int N, int Di, int Hi, int Wi, int C, void* cat, int ldc, int coff, int Do, int Ho,
                 int Wo, cudaStream_t stream);
int b2_upcat_bwd(const void* dcat, int ldc, int coff, int N, int Do, int Ho, int Wo, void* dx, int Di, int Hi,
                 int Wi, int C, cudaStream_t stream);

/* same result through two separable passes (W, then H/D) with a bf16 intermediate [N][Do][Ho][Wi][C] in `workspace`:
 * 2.3x fewer multiply-adds and loads than the single-pass gather                                                  */
long long b2_upcat_bwd_workspace_bytes(int N, int Do, int Ho, int Wi, int C);
int b2_upcat_bwd_separable(const void* dcat, int ldc, int coff, int N, int Do, int Ho, int Wo, void* dx, int Di,
                           int Hi, int Wi, int C, void* workspace, long long workspace_bytes, cudaStream_t stream);
int b2_upcat_bwd_separable_bstats(const void* dcat, int ldc, int coff, int N, int Do, int Ho, int Wo, void* dx,
                                  int Di, int Hi, int Wi, int C, void* workspace, long long workspace_bytes,
                                  const void* r, long long* stat_acc, cudaStream_t stream);

/* ---- final_conv 1x1x1 (pattern_class.py:364) fused with softmax / cross-entropy / argmax ------------------------ */
long long b2_head_workspace_bytes(int Cin);
/* loss_out[0] = mean CE over voxels with label >= 0 (NaN if none), loss_out[1] = sum; count_out = #labelled.
 * compute_grad: also d(loss)/d(x, W, b), scaled by grad_scale * (*grad_scale_dev if non-NULL).
 * eval_softmax: loss of Softmax outputs fed to CrossEntropyLoss, the reference's val-phase loss (training.py:189). */
/* x_scale_shift (fp32 [Cin][2], may be NULL; batch 1): x then holds the last layer's relu(conv) and its GroupNorm apply
 * y = bf16(r*scale + shift) is done on the gathered rows only, i.e. the dense apply pass over the volume is skipped */
int b2_head_ce(const void* x, const long long* labels, long long NV, const float* W, const float* b, int Cin,
               int Cout, float grad_scale, const float* grad_scale_dev, int compute_grad, int eval_softmax,
               int* preds, void* dx, float* dW, float* db, float* loss_out, int* count_out, void* workspace,
               long long workspace_bytes, const float* x_scale_shift, cudaStream_t stream);
/* training form (compute_grad, dx != NULL) that also accumulates the GroupNorm-backward statistics (sum dX, sum dX*r)
 * of the last trunk layer into stat_acc int64 [Cin][4]; r = that layer's saved relu(conv), dense bf16 [NV][Cin]     */
int b2_head_ce_bstats(const void* x, const long long* labels, long long NV, const float* W, const float* b, int Cin,
                      int Cout, float grad_scale, const float* grad_scale_dev, int* preds, void* dx, float* dW,
                      float* db, float* loss_out, int* count_out, void* workspace, long long workspace_bytes,
                      const void* r, long long* stat_acc, const float* x_scale_shift, int skip_dx_memset,
                      cudaStream_t stream);   /* skip_dx_memset: only the labelled rows of dx are written; pass the
                                                 labels to b2_relu_gn_bwd_acc (dy_row_labels) so the rest reads as 0 */
int b2_head_gather(const void* x, const long long* index, long long nidx, const float* W, const float* b, int Cin,
                   int Cout, int softmax, float* scores, int* preds, const float* x_scale_shift, cudaStream_t stream);
int b2_head_dense_fwd(const void* x, int N, long long V, const float* W, const float* b, int Cin, int Cout,
                      int softmax, float* out, cudaStream_t stream);
int b2_head_dense_bwd(const float* g, const void* x, int N, long long V, const float* W, int Cin, int Cout, void* dx,
                      float* dW, float* db, void* workspace, long long workspace_bytes, cudaStream_t stream);

/* ---- optimiser (training.py:140, 212) and bf16 weight packs ------------------------------------------------------
 * params/grads/moms/numels are HOST arrays of `count` entries (device pointers / element counts).                */
int b2_sgd_step(float* const* params, const float* const* grads, float* const* moms, const long long* numels,
                int count, float lr, float momentum, float grad_scale, cudaStream_t stream);
int b2_pack_conv_weights(const float* w, void* wf, void* wd, int Cout, int Cin, cudaStream_t stream);
/* all layers whose master weights changed, one launch; the five arrays are HOST arrays of `count` entries          */
int b2_pack_conv_weights_multi(const float* const* w, void* const* wf, void* const* wd, const int* cout,
                               const int* cin, int count, cudaStream_t stream);

/* ---- SulciDataset.__getitem__ on the device (SURVEY.md §8 f-1; reference dataset.py:66-88) ------------------------
 * point list (int32 [n][3] voxel coordinates + int32 [n] label ids) -> x fp32 [D][H][W] (1 at the points) and labels
 * int64 [D][H][W] (background elsewhere); duplicate points: the LAST one of the list wins, like the reference's CPU
 * index_put — bit-identical volumes.                                                                                 */
long long b2_scatter_volume_workspace_bytes(int D, int H, int W);
int b2_scatter_volume(const int* pts, const int* point_labels, int n, int D, int H, int W, float* x,
                      long long* labels, long long background, void* workspace, long long workspace_bytes,
                      cudaStream_t stream);
/* same with the rotation augmentation (dataset.py:33-43, 304-326) applied on the device: base_pts = the subject's
 * resident point list minus its minimum; xform = HOST double [12], R (row major) then t, built by the host from the
 * reference's random draws; the points scattered are trunc(R p + t) - min.  oob: device int32 [1], += number of
 * points outside the volume (the reference raises IndexError there; the host checks once per phase).                */
long long b2_scatter_volume_rot_workspace_bytes(int n, int D, int H, int W);
int b2_scatter_volume_rot(const int* base_pts, const int* point_labels, int n, const double* xform, int D, int H,
                          int W, float* x, long long* labels, long long background, int* oob, void* workspace,
                          long long workspace_bytes, cudaStream_t stream);

/* ---- post-inference integer pass: cutting(yscores, vert_notcut, bck2, threshold) (pattern_class.py:230) ---------
 * fold: dense ids in [0,F); thresholds: device int32 [T]; out: int32 [T][n].                                      */
long long b2_fold_vote_workspace_bytes(long long n, int C, int F, int T);
int b2_fold_vote(const float* scores, const int* fold, long long n, int C, int F, const int* thresholds, int T,
                 int* out, void* workspace, long long workspace_bytes, cudaStream_t stream);
/* test_thresholds() voxel matching (pattern_class.py:205-228): pts_a / pts_b int32 [n][3] = the native coordinates of
 * the same voxel set in the cut / not-cut graph order (|coordinate| < 2^20); out_a[i] = val_b[j] for the voxels i, j
 * of equal rank in the stable (x, y, z) sort of the two lists (the reference sorts both with pandas and zips).       */
long long b2_match_voxels_workspace_bytes(int n);
int b2_match_voxels(const int* pts_a, const int* pts_b, const int* val_b, int n, int* out_a, void* workspace,
                    long long workspace_bytes, cudaStream_t stream);
/* esi_score counters (training.py:223): counts uint64 [3][C] = TP, FP, FN, accumulated                            */
int b2_esi_counts(const int* y_true, const int* y_pred, long long n, int C, unsigned long long* counts,
                  cudaStream_t stream);
/* per-step epoch metrics of the batch loop (training.py:215-225) without leaving the device: labels int64 [n] (-1 =
 * unlabelled), preds int32 [n] (head kernel output) -> counts += TP/FP/FN; loss (fp32 device scalar, may be NULL):
 * loss_acc double [2] += {loss * loss_weight, loss_weight}.  One launch, capturable in the step's CUDA graph.        */
int b2_step_metrics(const long long* labels, const int* preds, long long n, int C, unsigned long long* counts,
                    const float* loss, double loss_weight, double* loss_acc, cudaStream_t stream);

/* ---- exact-label inference mode (labeling(), pattern_class.py:262-277, with fp32-accurate scores) ------------------
 * fp32 activations throughout; every 3x3x3 conv runs on b2_conv3d_igemm (y_is_fp32 = 1) over split operands:
 * b2_exact_split3 turns an fp32 channel window [V][C] into bf16 [V][3C] = [hi | lo | hi] (hi = bf16(x), lo =
 * bf16(x - hi)), paired with weights packed as [w_hi | w_hi | w_lo]: x*w to 2^-16 relative with fp32 accumulation.
 * b2_exact_split_first does the same for the binary network input: bf16 [V][32] = [x, x, 0 ...] against
 * [w_hi, w_lo, 0 ...].  The remaining operators are fp32: GroupNorm with fp64 statistics (deterministic two-stage
 * reduction; scale_shift fp32 [C][2]), MaxPool3d(2), trilinear upsample (align_corners=False) into a concat window,
 * and the 1x1x1 head + Softmax + arg-max at gathered voxels.  All tensors NDHWC, one sample.                        */
int b2_exact_split3(const float* x, long long V, int C, int ldx, int xoff, void* out, cudaStream_t stream);
int b2_exact_split_first(const float* x, long long V, void* out, cudaStream_t stream);
long long b2_exact_gn_workspace_bytes(int C);
int b2_exact_gn_stats(const float* r, long long V, int C, int G, float eps, const float* gamma, const float* beta,
                      float* scale_shift, void* workspace, long long workspace_bytes, cudaStream_t stream);
int b2_exact_gn_apply(const float* r, long long V, int C, const float* scale_shift, float* y, int ldy, int yoff,
                      cudaStream_t stream);
int b2_exact_maxpool(const float* x, int N, int D, int H, int W, int C, int ldx, int xoff, float* y,
                     cudaStream_t stream);
int b2_exact_upsample(const float* x, int N, int Di, int Hi, int Wi, int C, float* y, int ldy, int yoff, int Do, int Ho,
                      int Wo, cudaStream_t stream);
int b2_exact_head_gather(const float* x, const long long* index, long long n, const float* W, const float* b, int Cin,
                         int Cout, int softmax, float* scores, int* preds, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* UNETSULC_B200_H_ */
