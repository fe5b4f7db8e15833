/* b200seg.h -- C ABI of the B200-native segmentation hot path (libb200seg.so).
 *
 * Drop-in boundary for ONE path of taintpro98/rnd-semantic-segmentation: the DeepLabV2 ASPP
 * classifier head, align-corners upsample fused with (hard / soft-label) cross-entropy, and the
 * eval argmax + confusion-matrix.  The reference is pure Python/PyTorch and has no FFI of its own;
 * each entry point below names the reference call (file:line under the reference root) whose
 * arithmetic it replaces, and INTEGRATION.md shows the ctypes stubs a maintainer binds them with.
 *
 * Conventions
 *  - plain pointers and sizes only; every data pointer is a DEVICE pointer unless the name ends in
 *    "_host"; tensors are contiguous, fp32 NCHW / int64 NHW exactly as the reference passes them;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *    enqueued asynchronously on it, no hidden synchronisation, no hidden allocation: scratch is
 *    caller-provided and sized by the *_bytes() queries;
 *  - return value 0 = success; non-zero = error, message via b200seg_last_error() (thread-local);
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef B200SEG_H_
#define B200SEG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SEG_ABI_VERSION 1
#if defined(__GNUC__)
#define B200SEG_API __attribute__((visibility("default")))
#else
#define B200SEG_API
#endif

B200SEG_API int b200seg_abi_version(void);
B200SEG_API const char* b200seg_last_error(void);
/* number of SMs of the current device (148 on B200); <0 on error */
B200SEG_API int b200seg_device_sms(void);

/* ---------------------------------------------------------------------------------------------
 * K4  eval: upsample -> argmax(softmax) -> confusion matrix
 *   replaces  F.interpolate(align_corners=True) + F.softmax   core/utils/utility.py:185-186
 *             output.max(1)[1]                                 core/testers/aspp_tester.py:63
 *             confusion_matrix(cfg, pd, gt)                    core/utils/utility.py:347-359
 *   logits [N,C,h,w] f32; labels [N,H,W] i64 (may be NULL if cm is NULL);
 *   cm: i64, ACCUMULATED into; frame n adds into cm + n*cm_frame_stride (0 => one shared [C,C]);
 *   pred: optional i64 [N,H,W] argmax labels (bit-exact with the reference on CUDA);
 *   fma_mode: 0 = default (matches ATen's compiled expression); 1..3 = diagnostic variants.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_upsample_argmax_confusion(const float* logits, int N, int C, int h, int w, const int64_t* labels, int H,
                                      int W, int ignore_index, int64_t* cm, int64_t cm_frame_stride, int64_t* pred,
                                      int fma_mode, void* stream);

/* The same kernel with label / prediction maps in either element width -- label_bytes / pred_bytes = 8 (int64, what the
 * reference passes after `.long()`, core/testers/aspp_tester.py:58) or 1 (uint8, the tensor the dataloader already holds,
 * core/datasets/transform.py:31-33; SURVEY.md 8f rank 2): 8x fewer label bytes, no conversion pass. */
B200SEG_API int b200seg_upsample_argmax_confusion_ex(const float* logits, int N, int C, int h, int w, const void* labels,
                                         int label_bytes, int H, int W, int ignore_index, int64_t* cm, int64_t cm_frame_stride,
                                         void* pred, int pred_bytes, int fma_mode, void* stream);
/* Several frames of the tester loop (core/testers/aspp_tester.py:57-72, TEST.BATCH_SIZE = 1) in ONE launch: per-frame device
 * pointers in HOST arrays (logits_host[f] -> f32 [C,h,w]; labels_host[f] -> [H,W]; pred_host[f] -> [H,W] or pred_host NULL).
 * Any number of frames (16 per kernel launch).  cm as above (stride 0: one matrix for all frames). */
B200SEG_API int b200seg_upsample_argmax_confusion_frames(const float* const* logits_host, int n_frames, int C, int h, int w,
                                             const void* const* labels_host, int label_bytes, int H, int W, int ignore_index,
                                             int64_t* cm, int64_t cm_frame_stride, void* const* pred_host, int pred_bytes,
                                             void* stream);

/* confusion matrix from a materialised prediction map (API-compat form of utility.py:347-359);
 * mutate_pd != 0 also writes pd[i] = ignore_index where gt[i] == ignore_index, as
 * intersectionAndUnionGPU does to its `output` argument (utility.py:154). */
B200SEG_API int b200seg_confusion_from_pred(int64_t* pd, const int64_t* gt, int64_t n, int C, int ignore_index, int mutate_pd,
                                int64_t* cm, void* stream);
/* ... with int64 or uint8 maps (pd_bytes / gt_bytes = 8 or 1, any combination) */
B200SEG_API int b200seg_confusion_from_pred_ex(void* pd, int pd_bytes, const void* gt, int gt_bytes, int64_t n, int C,
                                   int ignore_index, int mutate_pd, int64_t* cm, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  upsample + softmax cross-entropy (ignore_index) forward, gradient w.r.t. low-res logits
 *   replaces  F.interpolate(...)                         core/models/classifiers/aspp/classifier.py:30-31
 *             .div(temperature)                          core/combos/aspp_fada.py:93-94
 *             CrossEntropyLoss(ignore_index=255)(o, y)   core/trainers/aspp_trainer.py:61,91
 *             loss.backward()                            core/trainers/aspp_trainer.py:92
 *   loss_out2: float[2] = { mean loss over valid pixels (NaN if none), number of valid pixels }.
 *   forward with need_grad != 0 leaves per-tile partial gradients in `workspace`; backward turns
 *   them into grad_logits [N,C,h,w] scaled by grad_out[0] (device scalar, NULL => 1).
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int64_t b200seg_upsample_ce_workspace_bytes(int N, int C, int h, int w, int H, int W);
B200SEG_API int b200seg_upsample_ce_forward(const float* logits, int N, int C, int h, int w, const int64_t* labels, int H, int W,
                                int ignore_index, float inv_temperature, int need_grad, void* workspace,
                                int64_t workspace_bytes, float* loss_out2, void* stream);
/* ... with int64 or uint8 labels (label_bytes = 8 or 1; the trainer's `.long()` at core/trainers/aspp_trainer.py:86 becomes
 * unnecessary: the uint8 tensor of core/datasets/transform.py:31-33 is consumed as it is) */
B200SEG_API int b200seg_upsample_ce_forward_ex(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes,
                                   int H, int W, int ignore_index, float inv_temperature, int need_grad, void* workspace,
                                   int64_t workspace_bytes, float* loss_out2, void* stream);
B200SEG_API int b200seg_upsample_ce_backward(const void* workspace, int N, int C, int h, int w, int H, int W,
                                 float inv_temperature, const float* loss_out2, const float* grad_out,
                                 float* grad_logits, void* stream);

/* K2 has two kernels with one contract: 1 (default) = the warp-tile kernel (csrc/ce_v2_kernels.cu) where it is eligible
 * (upsampling by >= ~5.3x horizontally, not downsampling vertically) and measured faster (19 classes); 2 = the warp-tile kernel
 * wherever it is eligible (19 or 2 classes); 0 = always the CTA-tile kernel (A/B experiments, cross-check in the tests). */
B200SEG_API void b200seg_upsample_ce_set_variant(int variant);

/* Packed backward for the fused head+loss path: writes the low-res gradient as bf16 class planes gOt [N][C][h*w]
 * (the NCHW layout at half the bytes; the buffer must hold N*h*w*32 elements) -- the operand layout
 * b200seg_aspp_backward_packed consumes -- and, if bias_grad != NULL, the per-class sum of the fp32 gradient
 * (= d loss / d bias of every ASPP branch).  No fp32 NCHW gradient is materialised. */
B200SEG_API int b200seg_upsample_ce_backward_packed(void* workspace, int N, int C, int h, int w, int H, int W,
                                        float inv_temperature, const float* loss_out2, const float* grad_out, void* gOt,
                                        float* bias_grad, void* stream);

/* materialising align-corners bilinear upsample and its adjoint ([NC,h,w] <-> [NC,H,W], f32)
 *   replaces  F.interpolate(..., mode='bilinear', align_corners=True)   classifier.py:31, discriminator.py:49 */
B200SEG_API int b200seg_upsample_bilinear_forward(const float* in, float* out, int NC, int h, int w, int H, int W, int fma_mode,
                                      void* stream);
B200SEG_API int b200seg_upsample_bilinear_backward(const float* grad_out, float* grad_in, int NC, int h, int w, int H, int W,
                                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3  soft-label cross-entropy on materialised [N,K,H,W] f32 operands
 *   replaces  soft_label_cross_entropy(pred, soft_label, pixel_weights)   core/utils/utility.py:172-177
 *   weights: optional [N,H,W] f32 (NULL => none).  loss_out: float[1].
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int64_t b200seg_soft_ce_workspace_bytes(void);
B200SEG_API int b200seg_soft_ce_forward(const float* pred, const float* soft, const float* weights, int N, int K, int H, int W,
                            void* workspace, int64_t workspace_bytes, float* loss_out, void* stream);
B200SEG_API int b200seg_soft_ce_backward(const float* pred, const float* soft, const float* weights, const float* grad_out, int N,
                             int K, int H, int W, float* grad_pred, void* stream);
/* Same loss, with the forward saving per-pixel statistics {log-sum-exp, sum_k q_k} (two f32 planes [N*H*W], needs
 * H*W % 4 == 0 and 16-byte aligned tensors) so that the backward is ONE 128-bit-vectorised streaming pass
 * (12*K + 8 bytes per pixel) instead of recomputing the softmax normaliser from a second read. */
B200SEG_API int64_t b200seg_soft_ce_stats_bytes(int N, int H, int W);
B200SEG_API int b200seg_soft_ce_forward_stats(const float* pred, const float* soft, const float* weights, int N, int K, int H, int W,
                                  void* workspace, int64_t workspace_bytes, float* stats, float* loss_out, void* stream);
B200SEG_API int b200seg_soft_ce_backward_stats(const float* pred, const float* soft, const float* weights, const float* stats,
                                   const float* grad_out, int N, int K, int H, int W, float* grad_pred, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5  FADA PixelDiscriminator loss tail, fused on low-resolution tensors
 *   replaces  F.interpolate(cat(cls1, cls2), size, align_corners=True)     core/models/discriminator.py:47-49
 *             softmax(seg_pred / T).detach(); soft[soft > 0.9] = 0.9        core/combos/aspp_fada.py:93-94,99-100,104-108
 *             cat((soft, 0)) [slot 0]  /  cat((0, soft)) [slot 1]           core/combos/aspp_fada.py:111,120,124
 *             soft_label_cross_entropy(D_pred, soft_label) + backward       core/utils/utility.py:172-177
 *   d_logits [N,2C,h,w] f32 (low-res discriminator output), seg_logits [N,C,h,w] f32 (low-res head output, treated
 *   as constant like the reference's .detach()).  loss_out2 = { loss, N*H*W }.  grad_d_logits [N,2C,h,w] f32.
 *   Any C <= 32: compile-time instantiations for C == 19 (Cityscapes/GTA5) and C == 2 (Kvasir/BLI), padded ones (8 / 16 / 24 / 32) otherwise.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int64_t b200seg_fada_softce_workspace_bytes(int N, int C, int h, int w, int H, int W);
B200SEG_API int b200seg_fada_softce_forward(const float* d_logits, const float* seg_logits, int N, int C, int h, int w, int H, int W,
                                float inv_temperature, float clamp, int slot, int need_grad, void* workspace,
                                int64_t workspace_bytes, float* loss_out2, void* stream);
B200SEG_API int b200seg_fada_softce_backward(const void* workspace, int N, int C, int h, int w, int H, int W,
                                 const float* loss_out2, const float* grad_out, float* grad_d_logits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K1  fused multi-dilation ASPP head (tcgen05 tap-packed GEMMs)
 *   replaces  ASPP_Classifier_V2.forward (size=None part)   core/models/classifiers/aspp/classifier.py:26-29
 *   R dilation branches (padding == dilation), weights R x [C,Cin,3,3] f32, biases R x [C] f32.
 *   NJ = b200seg_aspp_packed_rows(C, R): rows of the packed weight matrix ((8R+1)*C rounded to 128).
 *   Packed operands are bf16:  Wp [NJ,Cin], WpT [Cin,NJ], Xp [N*h*w, Cin].
 *   `weights`/`biases`/`grad_w`/`grad_b` are HOST arrays of R device pointers.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_aspp_packed_rows(int C, int R);
B200SEG_API int b200seg_aspp_pack_weights(const float* const* weights, const float* const* biases, int R, int C, int Cin, void* Wp,
                              void* WpT, float* bias_sum, void* stream);
B200SEG_API int b200seg_aspp_pack_features(const float* x_nchw, int N, int Cin, int h, int w, void* Xp, void* stream);
B200SEG_API int64_t b200seg_aspp_forward_scratch_bytes(int N, int C, int h, int w, int R);
B200SEG_API int b200seg_aspp_forward(const void* Xp, const void* Wp, const float* bias_sum, const int* rates_host, int R, int N,
                         int Cin, int C, int h, int w, void* scratch, float* logits, void* stream);
/* The same forward straight from the reference's fp32 NCHW features x [N,Cin,h,w] (classifier.py:26-29): the fp32 -> bf16
 * conversion of the pixel operand happens inside the GEMM's producer warps -- no b200seg_aspp_pack_features pass, no packed copy.
 * xn_bf16_nchw (optional, [N,Cin,h,w] bf16): a copy of the rounded features for the backward pass's weight-gradient GEMM.
 * Eligible shapes (b200seg_aspp_forward_f32_supported != 0): h*w % 4 == 0, Cin % 64 == 0, at least two 128-row tiles of packed
 * weights (e.g. 19 classes), x 16-byte aligned; otherwise returns an error and the caller packs. */
B200SEG_API int b200seg_aspp_forward_f32_supported(const float* x, int Cin, int C, int h, int w, int R);
B200SEG_API int b200seg_aspp_forward_f32(const float* x, const void* Wp, const float* bias_sum, const int* rates_host, int R, int N,
                                         int Cin, int C, int h, int w, void* scratch, float* logits, void* xn_bf16_nchw, void* stream);
B200SEG_API int64_t b200seg_aspp_backward_scratch_bytes(int N, int Cin, int C, int h, int w, int R, int splits);
/* grad_x (f32 NCHW, may be NULL), grad_w[r] / grad_b[r] (may be NULL) are overwritten, not accumulated */
B200SEG_API int b200seg_aspp_backward(const float* grad_logits, const void* Xp, const void* WpT, const int* rates_host, int R, int N,
                          int Cin, int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits, float* grad_x,
                          float* const* grad_w, float* const* grad_b, void* stream);

/* same as b200seg_aspp_backward but from the packed bf16 gradient planes gOt [N][C][h*w] (bias gradient comes
 * from b200seg_upsample_ce_backward_packed) */
B200SEG_API int b200seg_aspp_backward_packed(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N,
                                 int Cin, int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits,
                                 float* grad_x, float* const* grad_w, void* stream);

/* Seam-format variant (SURVEY.md section 8f rank 2: the backbone hands over bf16 channels_last features): the feature
 * gradient is written as bf16 pixel-major [N*h*w][Cin] (= NHWC / channels_last), half the bytes of the fp32 NCHW
 * gradient, by the same tcgen05 kernel with a bf16 epilogue.  Xp is then the backbone's own output, zero-copy. */
B200SEG_API int b200seg_aspp_backward_packed_nhwc(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N,
                                      int Cin, int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits,
                                      void* grad_x_nhwc_bf16, float* const* grad_w, void* stream);

/* Superset of the two entries above.  The weight gradients are computed FIRST; `weights_ready_event` (a cudaEvent_t,
 * may be NULL) is recorded on `stream` as soon as they are complete, before the data-gradient GEMM is enqueued, so a
 * data-parallel caller can run their NCCL all-reduce on a second stream underneath the data-gradient GEMM
 * (DDP semantics of train_distill.py:54-62).  Give at most one of grad_x (fp32 NCHW) / grad_x_nhwc_bf16. */
B200SEG_API int b200seg_aspp_backward_packed_ex(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N,
                                    int Cin, int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits, float* grad_x,
                                    void* grad_x_nhwc_bf16, float* const* grad_w, void* weights_ready_event, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K1 + K2 as ONE call per direction: the fused train slice
 *   replaces  pred = classifier(feat, size); loss = CrossEntropyLoss(ignore_index)(pred / T, label); loss.backward()
 *             core/trainers/aspp_trainer.py:86-93, core/combos/aspp_fada.py:88-96  (head: core/models/classifier.py:26-31)
 *   forward : pack weights -> pack features (x_kind 0) -> 33-tap GEMM -> gather + bias -> upsample + CE (+ gradient partials) -> loss
 *   backward: low-res gradient (bf16 planes) + bias gradients -> G't -> weight-gradient GEMM -> reduce -> [event] -> data-gradient GEMM
 * The host cost of the step is the enqueue of these ~12 kernels; one foreign call each way keeps 1-2 image batches GPU-bound.
 *   x        x_kind 0: fp32 NCHW [N,Cin,h,w];  x_kind 1: bf16 pixel-major [N*h*w, Cin] (channels_last seam format, used in place)
 *   workspace  b200seg_head_loss_workspace_bytes(...) bytes, owned by the caller from forward until backward has run
 *   scratch    b200seg_head_loss_scratch_bytes(...) bytes, transient inside each call (stream-ordered reuse is fine)
 *   logits   fp32 [N,C,h,w] (out),  loss_out fp32 [1] (out; NaN when every label is ignored, like the reference)
 *   backward: grad_loss fp32 [1] or NULL (= 1); give at most one of grad_x (fp32 NCHW) / grad_x_nhwc_bf16; grad_w / grad_b are
 *   R pointers each (or NULL; every branch bias receives the same gradient); weights_ready_event as in
 *   b200seg_aspp_backward_packed_ex.  x_bf16 = the forward's x when x_kind == 1 (the caller keeps it alive), else NULL.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int64_t b200seg_head_loss_workspace_bytes(int N, int Cin, int C, int h, int w, int R, int H, int W, int x_kind);
B200SEG_API int64_t b200seg_head_loss_scratch_bytes(int N, int Cin, int C, int h, int w, int R);
B200SEG_API int b200seg_head_loss_forward(const void* x, int x_kind, const float* const* weights, const float* const* biases,
                                    const int* rates_host, int R, int N, int Cin, int C, int h, int w, const void* labels,
                                    int label_bytes, int H, int W, int ignore_index, float inv_temperature, int need_grad,
                                    void* workspace, int64_t workspace_bytes, void* scratch, int64_t scratch_bytes, float* logits,
                                    float* loss_out, void* stream);
B200SEG_API int b200seg_head_loss_backward(void* workspace, int64_t workspace_bytes, const void* x_bf16, int x_kind,
                                    const int* rates_host, int R, int N, int Cin, int C, int h, int w, int H, int W,
                                    float inv_temperature, const float* grad_loss, void* scratch, int64_t scratch_bytes,
                                    float* grad_x, void* grad_x_nhwc_bf16, float* const* grad_w, float* const* grad_b,
                                    void* weights_ready_event, void* stream);
/* The two entries above replay their kernel sequence from a CUDA graph once the same arguments (addresses, shapes, scalars) have
 * been seen twice -- a training loop in steady state gets the same addresses back from its allocator every iteration, and ~7
 * launches per direction become one cudaGraphLaunch on the caller's stream (weights_ready_event is recorded from inside the
 * graph as an external event node).  Direct launches whenever the caller is itself capturing, per-kernel profiling is on, or the
 * addresses keep changing (the cache then turns itself off).  on = 0 disables (also env B200SEG_STEP_GRAPHS=0); stats: replays
 * and captures so far. */
B200SEG_API void b200seg_set_step_graphs(int on);
B200SEG_API void b200seg_step_graph_stats(long long* replays, long long* captures);
/* split-K factor the weight-gradient GEMM uses for P = N*h*w pixels (what the entries above pick) */
B200SEG_API int b200seg_aspp_default_wgrad_splits(int64_t P, int C, int Cin, int R);

/* ---------------------------------------------------------------------------------------------
 * K6  3x3 convolution layers as tcgen05 implicit GEMMs: the PixelDiscriminator conv stack
 *   replaces  D = Conv2d(Cin,ndf,3,1,1)+LeakyReLU(0.2)+Conv2d(ndf,ndf/2,3,1,1)+LeakyReLU(0.2)   core/models/discriminator.py:34-39
 *             cls1 / cls2 = Conv2d(ndf/2, C, 3, 1, 1)                                            core/models/discriminator.py:40-41
 *             their application and torch.cat                                                   core/models/discriminator.py:45-47
 *             and the autograd backward of those layers (call sites core/trainers/aspp_fada.py:110,119,123)
 *   Activations are bf16 NHWC [N,h,w,pitch] (pitch = channels rounded to a multiple of 8); weights are packed once per
 *   parameter update.  Stride 1, padding == dilation.  The zero padding is the TMA unit's out-of-bounds fill.
 * ------------------------------------------------------------------------------------------- */
/* The whole stack in ONE call per direction (replayed from a CUDA graph once the same arguments have been seen twice, like
 * b200seg_head_loss_forward / _backward; every buffer is caller-provided, results bit-identical to the separate entries below):
 *   forward : [pack w1, w2, cls1 | cls2 (do_pack)] -> [pack x (x_kind 0: fp32 NCHW; 1: bf16 NHWC used in place)] -> conv + LReLU ->
 *             conv + LReLU -> cls1 | cls2 -> out fp32 [N, 2C, h, w]                     discriminator.py:34-47
 *   backward: grad_out fp32 [N, 2C, h, w] -> bf16 NHWC -> bias / weight / data gradients of the three layers (LeakyReLU' fused
 *             into the data-gradient epilogues); NULL outputs are skipped together with everything only they need
 *   Wf_l / Wb_l: bf16 [9][Co_l][Ci_l] / [9][Ci_l][round8(Co_l)]; b3 fp32 [2C]; Xp / A1 / A2 / G3 / dZ2 / dZ1: bf16 NHWC;
 *   gb3 fp32 [2C] = the cls1 | cls2 bias gradients; scratch: b200seg_disc_backward_scratch_bytes(...) bytes */
B200SEG_API int b200seg_disc_forward(const void* x, int x_kind, int N, int Cin, int h, int w, int ndf1, int ndf2, int C,
                                    const float* w1, const float* b1, const float* w2, const float* b2, const float* wc1,
                                    const float* bc1, const float* wc2, const float* bc2, float slope, int do_pack, void* Wf1,
                                    void* Wb1, void* Wf2, void* Wb2, void* Wf3, void* Wb3, float* b3, void* Xp, void* A1, void* A2,
                                    float* out, void* stream);
B200SEG_API int64_t b200seg_disc_backward_scratch_bytes(int N, int Cin, int h, int w, int ndf1, int ndf2, int C);
B200SEG_API int b200seg_disc_backward(const float* grad_out, const void* Xp, const void* A1, const void* A2, const void* Wb1,
                                    const void* Wb2, const void* Wb3, int N, int Cin, int h, int w, int ndf1, int ndf2, int C,
                                    float slope, void* G3, void* dZ2, void* dZ1, void* scratch, int64_t scratch_bytes, float* gw1,
                                    float* gb1, float* gw2, float* gb2, float* gwc1, float* gwc2, float* gb3, float* gx_f32_nchw,
                                    void* gx_bf16_nhwc, void* stream);
/* n_parts weight tensors fp32 [part_co[i]][Ci][3][3], concatenated along the output-channel axis (cls1 | cls2 = torch.cat(dim=1)):
 *   Wf bf16 [9][Co][Ci]        forward operand (Co = sum part_co)           (may be NULL)
 *   Wb bf16 [9][Ci][co_pitch]  data-gradient operand, caller zero-fills the padding columns co_pitch > Co   (may be NULL) */
B200SEG_API int b200seg_conv3x3_pack_weights(const float* const* weights, const int* part_co_host, int n_parts, int Ci, void* Wf,
                                             void* Wb, int co_pitch, void* stream);
/* the same for a whole stack of layers in ONE launch (training re-packs every step): layer l owns parts_per_layer[l] consecutive
 * entries of weights / part_co (all HOST arrays; weights holds device pointers), writes Wf[l] / Wb[l] (either may be NULL) with
 * row pitch co_pitch[l]; the padding columns of every Wb are zero-filled by the kernel.  bias_parts (n_bias <= 4 device pointers,
 * NULL = zeros, lengths bias_len) are concatenated into bias_out -- the cls1 | cls2 bias of discriminator.py:39-40,47 */
B200SEG_API int b200seg_conv3x3_pack_weights_stack(int n_layers, const float* const* weights, const int* part_co_host,
                                                   const int* parts_per_layer_host, const int* Ci_host, void* const* Wf, void* const* Wb,
                                                   const int* co_pitch_host, const float* const* bias_parts, const int* bias_len_host,
                                                   int n_bias, float* bias_out, void* stream);
/* out = [LeakyReLU_slope](conv3x3(act; Wf) + bias): exactly one of out_bf16_nhwc ([N,h,w,out_pitch]) / out_f32_nchw ([N,Co,h,w]);
 * bias may be NULL; lrelu != 0 applies the activation */
B200SEG_API int b200seg_conv3x3_forward(const void* act_nhwc_bf16, int N, int h, int w, int Ci, int64_t act_pitch, const void* Wf, int Co,
                                        int dilation, const float* bias, int lrelu, float slope, void* out_bf16_nhwc,
                                        int64_t out_pitch, float* out_f32_nchw, void* stream);
/* gin = conv3x3_transposed(g; Wb) [* LeakyReLU'(mask)]: g bf16 NHWC [N,h,w,g_pitch] with Cg = the pitch of Wb's last axis;
 * mask (optional, bf16 NHWC, same layout as out_bf16_nhwc) is the saved post-activation output of the layer below:
 * the gradient is multiplied by 1 where mask > 0 and by slope elsewhere (LeakyReLU backward fused in the epilogue) */
B200SEG_API int b200seg_conv3x3_dgrad(const void* g_nhwc_bf16, int N, int h, int w, int Cg, int64_t g_pitch, const void* Wb, int Ci,
                                      int dilation, const void* mask_nhwc_bf16, float slope, void* out_bf16_nhwc, int64_t out_pitch,
                                      float* out_f32_nchw, void* stream);
/* the same data gradient (bf16 NHWC output only) that also returns colsum_out[ci] = sum_pixels out[pixel][ci] (fp32 [Ci]): the bias
 * gradient of the layer below (what autograd derives for discriminator.py:35,37's Conv2d biases), accumulated in the GEMM epilogue
 * from the stored (bf16-rounded) values and finished by one fixed-order reduction -- no second pass over the tensor */
B200SEG_API int64_t b200seg_conv3x3_dgrad_colsum_scratch_bytes(int N, int h, int w, int64_t out_pitch);
B200SEG_API int b200seg_conv3x3_dgrad_colsum(const void* g_nhwc_bf16, int N, int h, int w, int Cg, int64_t g_pitch, const void* Wb, int Ci,
                                             int dilation, const void* mask_nhwc_bf16, float slope, void* out_bf16_nhwc,
                                             int64_t out_pitch, void* colsum_scratch, int64_t colsum_scratch_bytes, float* colsum_out,
                                             void* stream);
/* grad_w[i] fp32 [part_co[i]][Ci][3][3] = sum_pixels g[pixel, co] * x[pixel + tap, ci]; splits <= 0 picks the split-K factor */
B200SEG_API int64_t b200seg_conv3x3_wgrad_scratch_bytes(int N, int h, int w, int Co, int Ci, int splits);
B200SEG_API int b200seg_conv3x3_wgrad(const void* g_nhwc_bf16, int Co, int64_t g_pitch, const void* x_nhwc_bf16, int Ci, int64_t x_pitch,
                                      int N, int h, int w, int dilation, int splits, void* scratch, int64_t scratch_bytes,
                                      float* const* grad_w, const int* part_co_host, int n_parts, void* stream);
/* fp32 NCHW [N,C,hw] -> bf16 NHWC [N*hw][pitch] (channels >= C zero): the output gradient of the last layer */
B200SEG_API int b200seg_nchw_to_nhwc_bf16(const float* src, int N, int C, int hw, void* dst, int pitch, void* stream);
/* bias gradient: out[c] = sum_pixels g[pixel][c], deterministic (fixed-order two-phase sum) */
B200SEG_API int64_t b200seg_nhwc_colsum_scratch_bytes(int pitch);
B200SEG_API int b200seg_nhwc_bf16_colsum(const void* g_nhwc_bf16, int64_t P, int C, int pitch, void* scratch, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Seam-format producer: the fused tail of the backbone's last Bottleneck (SURVEY 8f rank 2)
 * b200seg_seam_tail_forward  replaces  out = self.bn3(out); out += identity; out = self.relu(out)
 *                                      (core/models/feature_extractor/resnet.py:106-113, bn3 a FrozenBatchNorm2d: x * scale + bias,
 *                                      core/models/layers.py:17-23) and the bf16 channels_last cast the head's seam format takes:
 *   y bf16 NHWC [N][hw][C] = bf16_rn(relu((c * scale + bias) + identity)), c / identity fp32 NCHW [N][C][hw], scale / bias fp32 [C]
 *   (the folded norm).  Each step rounded in fp32 in that order, no FMA contraction: y is bit-identical to the stock output cast
 *   with .to(torch.bfloat16).
 * b200seg_seam_tail_backward  replaces  the autograd backward of the same lines:
 *   g = dy * (y > 0);  dc fp32 NCHW = g * scale;  didentity fp32 NCHW = g     (dy, y bf16 NHWC as above)
 *   dc or didentity may be NULL when that gradient is not wanted.
 * C % 8 == 0, any hw >= 1, any N; y and dy 16-byte aligned.  No scratch.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_seam_tail_forward(const float* c, const float* identity, const float* scale, const float* bias, int N, int C,
                                          int hw, void* y, void* stream);
B200SEG_API int b200seg_seam_tail_backward(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc,
                                           float* didentity, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K7  test-time augmentation fused with argmax + confusion matrix (SURVEY 8f rank 3).
 * Replaces inference(..., flip=True) (core/utils/utility.py:179-191), multi_scale_inference (utility.py:193-209), the
 * output.max(1)[1] / output.argmax(0) that follow (core/testers/aspp_tester.py:63,42) and confusion_matrix /
 * intersectionAndUnionGPU (utility.py:347-359,148-161) for ONE frame:
 *   prob = (sum_m flip_m(softmax(upsample(logits_lr[m], (H,W))))) / divisors[0] [/ divisors[1]];  pred = first argmax(prob)
 * logits_lr: HOST array of n_members (<= 8) device pointers to fp32 [C, h[m], w[m]]; flip[m] != 0: the member was computed on
 * the horizontally mirrored image, its probabilities are mirrored back.  Members are summed in array order (the reference's
 * order: scale-major, plain before flipped).  div_exact = 0 multiplies by the fp32 reciprocal of each divisor (what ATen's CUDA
 * `tensor / python_scalar` does), 1 divides (ATen's CPU kernel).  Outputs, each optional (NULL): cm int64 [C,C] accumulated
 * into (rows = truth, needs labels int64 [H,W]; truth == ignore_index or outside [0,C) skipped), pred int64 [H,W], probs fp32
 * [C,H,W] (the tensor the reference returns).
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_tta_argmax_confusion(const float* const* logits_lr, const int* h, const int* w, const int* flip, int n_members,
                                             int C, const int64_t* labels, int H, int W, int ignore_index, const float* divisors,
                                             int n_div, int div_exact, int64_t* cm, int64_t* pred, float* probs, void* stream);
/* ... with int64 or uint8 label and prediction maps (label_bytes / pred_bytes = 8 or 1): uint8 labels as the dataloader holds them
 * (core/datasets/transform.py:31-33), uint8 predictions as the pseudo-label writer stores them (core/testers/aspp_tester.py:40-45) */
B200SEG_API int b200seg_tta_argmax_confusion_ex(const float* const* logits_lr, const int* h, const int* w, const int* flip,
                                                int n_members, int C, const void* labels, int label_bytes, int H, int W,
                                                int ignore_index, const float* divisors, int n_div, int div_exact, int64_t* cm,
                                                void* pred, int pred_bytes, float* probs, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Mean all-reduce of a flat fp32 gradient bucket over NVLink / NVSwitch peer memory (one kernel per rank)
 *   replaces  the gradient all-reduce of DistributedDataParallel      train_distill.py:54-62 (mean over ranks)
 *   The bucket lives in symmetric memory: peer_bufs_host[q] = rank q's bucket as mapped into THIS process, signal_pads_host[q] =
 *   rank q's signal pad (uint32 flags, all zero between calls), multicast_ptr = the bucket's NVSwitch multicast address or NULL
 *   (then plain peer loads / stores are used).  numel: bucket length in floats, a multiple of 4.  Every rank must enqueue the call
 *   (the kernels meet at two cross-rank barriers); `blocks` CTAs of 512 threads, using pad slots [pad_slot0, pad_slot0 + blocks).
 *   On return of the kernel every rank's bucket holds sum over ranks / world, bit-identical on all ranks.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_p2p_allreduce_mean(void* const* peer_bufs_host, void* multicast_ptr, void* const* signal_pads_host, int rank,
                                           int world, int64_t numel, int blocks, int pad_slot0, void* stream);

/* ensembles of up to four members: 1 (default) = the row-walking kernel (horizontal lerps of the two current source rows kept per
 * thread in shared memory and re-used for every output row between them), 0 = the per-pixel kernel used for larger ensembles
 * (A/B experiments; the results are bit-identical).  Bit 1 set (on = 3): row walking without the labels-only fast path (when no
 * probabilities are requested the kernel orders the classes with ex2.approx-based probabilities and re-runs ATen's exact
 * sequence only for pixels whose best two sums are within 2e-5 per member; labels and matrix stay bit-exact) */
B200SEG_API void b200seg_tta_set_row_walk(int on);

/* ---------------------------------------------------------------------------------------------
 * K8  multi-tensor optimizer steps (SURVEY 8f rank 4), one launch per group of <= 16 tensors.  The pointer arrays are HOST
 * arrays of device pointers, numels the element counts.  grad_scale multiplies every gradient as it is read (1/world_size after
 * a SUM all-reduce = DDP's mean, train_distill.py:54-62; 1.0f = off).
 * b200seg_sgd_step  = torch.optim.SGD(lr, momentum, dampening, weight_decay, nesterov).step()
 *                     (core/trainers/aspp_trainer.py:25-26,94-95); first_step != 0: the momentum buffers are uninitialised and
 *                     are set to the gradient (torch's momentum_buffer is None case); momentum_bufs may be NULL when momentum == 0.
 * b200seg_adam_step = torch.optim.Adam(lr, betas, eps, weight_decay).step() (core/adapters/fada_adapter.py:24), step = the
 *                     update count INCLUDING this one (>= 1); exp_avg / exp_avg_sq start at zero.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API int b200seg_sgd_step(int n_tensors, float* const* params, const float* const* grads, float* const* momentum_bufs,
                                 const int64_t* numels, float lr, float momentum, float dampening, float weight_decay, int nesterov,
                                 int first_step, float grad_scale, void* stream);
B200SEG_API int b200seg_adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                                  float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2, float eps,
                                  float weight_decay, int64_t step, float grad_scale, void* stream);

/* ---------------------------------------------------------------------------------------------
 * instrumentation (bench.py): number of kernels this library has launched, and per-kernel CUDA-event
 * timing on the launching stream.  Tags: 0 head fwd GEMM, 1 head dgrad GEMM, 2 head wgrad GEMM,
 * 3 feature pack, 4 fwd gather, 5 grad im2col (G'), 6 upsample+CE main, 7 eval argmax+confusion,
 * 8 soft-CE fwd, 9 soft-CE bwd, 10 wgrad reduce, 11 fused FADA soft-CE main, 12 conv3x3 fwd, 13 conv3x3 dgrad,
 * 14 conv3x3 wgrad, 15 test-time-augmentation argmax+confusion.
 * ------------------------------------------------------------------------------------------- */
B200SEG_API long long b200seg_launch_count(void);
B200SEG_API void b200seg_profile_enable(int on);
B200SEG_API int b200seg_profile_read(int tag, double* total_ms, int* count);

/* on-device self-test of the tcgen05 GEMM core against a CUDA-core reference (synchronous).
 * share: 0 = one CTA per tile, 1 = 2-CTA cluster multicasting the shared B tile, 2 = ... the shared A tile,
 *        3 = 2 x 2 cluster multicasting both, 4 = CTA pair on one tcgen05.mma.cta_group::2 (M = 256). */
B200SEG_API int b200seg_gemm_selftest(int M, int N, int K, int a_mn_major, int b_mn_major, int splits, int col_hw, int share,
                          double* max_err, double* max_ref);
/* head forward GEMM: 1 (default) = the tile width (256 / 224 / 192 accumulator columns) is chosen per problem so that the tile
 * count is a near-multiple of the SM count (wave quantisation), 0 = always 256 */
B200SEG_API void b200seg_gemm_set_narrow_tiles(int on);
/* fp32 NCHW data gradient of the head (the dX of classifier.py:26-29's convolutions): 0 = channels along the GEMM's M dimension
 * (shared-memory transpose epilogue), 1 (default) = pixels along M as CTA pairs, stored straight from the accumulator registers
 * (lane = pixel: one store instruction = 32 consecutive pixels of a channel plane; seven ring stages), 2 = the same
 * with streaming (evict-first) stores (measured no better).  The tile order of every GEMM follows the operand sizes (the larger
 * operand streams from HBM once). */
B200SEG_API void b200seg_gemm_set_dgrad_mode(int mode);
/* forward GEMM of the head (classifier.py:26-29): 0 = channel-major (M = packed weight rows; 5 M-tiles on 3 CTA pairs), 1 (default)
 * = pixel-major (M = pixels, the 2.5 N-tiles' ragged last one at half MMA width, register-store epilogue) */
B200SEG_API void b200seg_gemm_set_fwd_mode(int mode);
/* 1: the head's forward takes fp32 NCHW features through the GEMM with in-kernel conversion (below) where the shape is eligible;
 * 0 (default): pack + plain GEMM.  Measured equal at the eval shape (158.8 vs 158.3 us); kept as a tested option. */
B200SEG_API void b200seg_gemm_set_fwd_convert(int on);
/* on-device self-test of that kernel against a CUDA-core reference on bf16-rounded x; xn_err: max |bf16 copy - bf16(x)| */
B200SEG_API int b200seg_gemm_fwd_convert_selftest(int M, int n_img, int hw, int K, int write_xn, double* max_err, double* max_ref,
                                      double* xn_err);
/* K6 conv kernel: 1 (default) = CTA pairs driving one tcgen05.mma.cta_group::2 (M = 256) wherever a layer has two M-tiles,
 * 0 = one CTA per tile (A/B experiments) */
B200SEG_API void b200seg_conv_set_pair(int on);
/* operand sharing inside the ASPP head GEMMs: 0 none, 1 (default) 2-CTA multicast pairs, 2 2 x 2 clusters sharing both
 * operands, 3 = 1, plus cta_group::2 pairs (one 2-SM MMA) for the GEMMs whose pairs lie along M (the data gradient) */
B200SEG_API void b200seg_gemm_set_sharing(int on);
/* SMs the data-gradient GEMM leaves free when b200seg_aspp_backward_packed_ex is given a weights_ready_event, so that the
 * caller's all-reduce kernel can be resident underneath it (the persistent GEMM otherwise fills every SM's shared memory);
 * default 8 */
B200SEG_API void b200seg_gemm_set_overlap_sms(int n);

#ifdef __cplusplus
}
#endif
#endif /* B200SEG_H_ */
