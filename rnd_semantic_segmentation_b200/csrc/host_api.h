// Host functions defined in one translation unit and called from another, declared once.  Every defining file includes this
// header, so the compiler checks each definition against its declaration (the build also rejects a definition without a
// prior declaration, -Werror=missing-declarations).  Host-only: no device code, no gemm types (those stay in gemm_sm100.cuh).
#pragma once
#include <cuda_runtime.h>

namespace b200seg {

// ---- eval_kernels.cu ----
int k4_launch(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H, int W, int ignore_index,
              long long* cm, long long cm_frame_stride, void* pred, int pred_bytes, int fma_mode, cudaStream_t stream);
int k4_launch_frames(const float* const* logits, int n_frames, int C, int h, int w, const void* const* labels, int label_bytes, int H,
                     int W, int ignore_index, long long* cm, long long cm_frame_stride, void* const* pred, int pred_bytes, int fma_mode,
                     cudaStream_t stream);
int confusion_pairs_launch_ex(void* pd, int pd_bytes, const void* gt, int gt_bytes, long long n, int C, int ignore_index, int mutate_pd,
                              long long* cm, cudaStream_t stream);

// ---- ce_kernels.cu ----
void k2_set_variant(int v);           // A/B: 0 = always the CTA-tile kernel, 1 = warp-tile kernel where eligible (default)
long long k2_workspace_bytes(int N, int C, int h, int w, int H, int W);
int k2_forward(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H, int W, int ignore_index,
               float inv_T, int need_grad, void* workspace, long long workspace_bytes, float* loss_out2, cudaStream_t stream,
               float* loss_copy = nullptr);
int k2_backward(const void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                const float* grad_out, float* grad_logits, cudaStream_t stream);
int k2_backward_packed_multi(void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                             const float* grad_out, void* gOt, float* const* bias_grads, int n_bias, cudaStream_t stream);
int k2_backward_packed(void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                       const float* grad_out, void* gOt, float* bias_grad, cudaStream_t stream);
long long k5_workspace_bytes(int N, int C, int h, int w, int H, int W);
int k5_forward(const float* dlogits, const float* slogits, int N, int C, int h, int w, int H, int W, float inv_T, float clamp, int slot,
               int need_grad, void* workspace, long long workspace_bytes, float* loss_out2, cudaStream_t stream);
int k5_backward(const void* workspace, int N, int C, int h, int w, int H, int W, const float* loss_out2, const float* grad_out,
                float* grad_d, cudaStream_t stream);
int upsample_fwd_launch(const float* in, float* out, int NC, int h, int w, int H, int W, int fma_mode, cudaStream_t stream);
int upsample_bwd_launch(const float* gout, float* gin, int NC, int h, int w, int H, int W, cudaStream_t stream);

// ---- softce_kernels.cu ----
long long k3_workspace_bytes();
long long k3_stats_bytes(int N, int H, int W);
int k3_forward(const float* pred, const float* soft, const float* wts, int N, int K, int H, int W, void* workspace,
               long long workspace_bytes, float* loss_out, cudaStream_t stream, float* stats);
int k3_backward(const float* pred, const float* soft, const float* wts, const float* grad_out, int N, int K, int H, int W,
                float* grad_pred, cudaStream_t stream, const float* stats);

// ---- aspp_head.cu ----
int aspp_nj(int C, int R);
int aspp_pack_weights(const float* const* w, const float* const* b, int R, int C, int Cin, void* Wp, void* WpT, float* bias_sum,
                      cudaStream_t stream);
int aspp_pack_features(const float* x, int N, int Cin, int h, int w, void* Xp, cudaStream_t stream);
long long aspp_yt_bytes(int N, int C, int h, int w, int R);
int aspp_forward(const void* Xp, const void* Wp, const float* bias_sum, const int* rates, int R, int N, int Cin, int C, int h, int w,
                 float* Yt, float* logits, cudaStream_t stream);
int aspp_forward_f32_supported(const float* x, int Cin, int C, int h, int w, int R);
int aspp_forward_f32(const float* x, const void* Wp, const float* bias_sum, const int* rates, int R, int N, int Cin, int C, int h,
                     int w, float* Yt, float* logits, void* xn, cudaStream_t stream);
long long aspp_bwd_scratch_bytes(int N, int Cin, int C, int h, int w, int R, int splits);
void* aspp_bwd_gOt_ptr(void* scratch);
int aspp_backward_packed(const void* gOt_in, const void* Xp, const void* WpT, const int* rates, int R, int N, int Cin, int C, int h,
                         int w, void* scratch, long long scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                         cudaStream_t stream, void* grad_x_nhwc_bf16, cudaEvent_t weights_ready);
int aspp_backward(const float* grad_logits, const void* Xp, const void* WpT, const int* rates, int R, int N, int Cin, int C, int h,
                  int w, void* scratch, long long scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                  float* const* grad_b, cudaStream_t stream);

// ---- conv_sm100.cu ----
// tf32 != 0: the TF32 layers -- act / g / x / mask / Wf / Wb and the NHWC outputs are fp32 (TF32 values) instead of bf16
int conv3x3_pack_weights(const float* const* weights, const int* part_co, int n_parts, int Ci, void* Wf, void* Wb, int co_pitch,
                         cudaStream_t stream);
int conv3x3_pack_weights_stack(int n_layers, const float* const* weights, const int* part_co, const int* parts_per_layer,
                               const int* Ci, void* const* Wf, void* const* Wb, const int* co_pitch, const float* const* bias_parts,
                               const int* bias_len, int n_bias, float* bias_out, cudaStream_t stream);
int conv3x3_pack_weights_stack_tf32(int n_layers, const float* const* weights, const int* part_co, const int* parts_per_layer,
                                    const int* Ci, void* const* Wf, void* const* Wb, const int* co_pitch, const float* const* bias_parts,
                                    const int* bias_len, int n_bias, float* bias_out, cudaStream_t stream);
int conv3x3_forward(const void* act, int N, int h, int w, int Ck, long long act_pitch, const void* Wf, int Co, int dilation,
                    const float* bias, int lrelu, float slope, void* out_nhwc, long long out_pitch, float* out_f32_nchw,
                    cudaStream_t stream, int tf32 = 0);
// out_bf16_nhwc: with tf32 only, the layer's result as bf16 NHWC (the feature gradient of bf16 channels_last features)
int conv3x3_dgrad(const void* g, int N, int h, int w, int Cg, long long g_pitch, const void* Wb, int Ci, int dilation,
                  const void* mask, float slope, void* out_nhwc, long long out_pitch, float* out_f32_nchw, cudaStream_t stream,
                  void* colsum_scratch, long long colsum_scratch_bytes, float* colsum_out, int tf32 = 0, void* out_bf16_nhwc = nullptr);
long long conv3x3_dgrad_colsum_scratch_bytes(int N, int h, int w, long long out_pitch);
long long conv3x3_wgrad_scratch_bytes(int N, int h, int w, int Co, int Ci, int splits);
int conv3x3_wgrad(const void* g, int Co, long long g_pitch, const void* x, int Ci, long long x_pitch, int N, int h, int w,
                  int dilation, int splits, void* scratch, long long scratch_bytes, float* const* grad_w, const int* part_co,
                  int n_parts, cudaStream_t stream, int tf32 = 0);
long long nhwc_colsum_scratch_bytes(int pitch);
int nhwc_bf16_colsum(const void* g, long long P, int C, int pitch, void* scratch, float* out, cudaStream_t stream);
int nchw_channel_sum(const float* src, int N, int C, int hw, float* out, cudaStream_t stream);       // out[c] = sum src[n][c][:]
int widen_bf16(const void* src, long long n, float* dst, cudaStream_t stream);                       // bf16 [n] -> fp32 [n], exact
namespace gemm { namespace conv {
void set_pair(int on);                // 0 = one CTA per tile, 1 = CTA pairs (cta_group::2) where two M-tiles exist
} }

// ---- gemm_sm100.cu: host controls of the tcgen05 GEMM (launch() and the types it takes: gemm_sm100.cuh) ----
namespace gemm {
void set_sharing(int on);
void set_overlap_sms(int n);
int overlap_sms();                    // SMs the data-gradient GEMM leaves free while an all-reduce overlaps it
void set_narrow_tiles(int on);
// fp32 NCHW data gradient of the head: 0 = channels along M (shared-memory transpose epilogue), 1 = pixels along M as cta_group::2
// pairs, stores straight from registers, seven ring stages
void set_dgrad_mode(int mode);
int dgrad_mode();
// forward GEMM of the head: 0 = channel-major (M = packed weight rows, shared-memory transpose epilogue), 1 = pixel-major
// (M = pixels, register stores, ragged last N-tile at half MMA width)
void set_fwd_mode(int mode);
int fwd_mode();
void set_fwd_convert(int on);
int selftest(int M, int N, int K, int a_mn, int b_mn, int splits, int col_hw, int share, double* max_err, double* max_ref);
int selftest_fwd_convert(int M, int n_img, int hw, int K, int write_xn, double* max_err, double* max_ref, double* xn_err);
int run(const void* a, int a_mn, long long a_pitch, const void* b, int b_mn, long long b_pitch, int M, int N, int K, int layout,
        void* out, long long row_stride, long long img_stride, long long split_stride, int hw, const float* identity,
        const float* scale, const float* bias, void* stats, int splits, int share, int pair_fallback, int sm_reserve,
        int* splits_used, int* variant, cudaStream_t stream);
// the kernels launch() chooses from: their count, and entry i's template arguments (B200SEG_ERR_ARG for i out of range)
int variant_count();
int variant_info(int i, int* a_mn, int* b_mn, int* share, int* bn, int* rs, int* seam, int* stats);
}  // namespace gemm

// ---- seam_tail_kernels.cu ----
int seam_tail_forward(const float* c, const float* identity, const float* scale, const float* bias, int N, int C, int hw, void* y,
                      cudaStream_t stream);
int nchw_to_nhwc_bf16(const float* src, int N, int C, int hw, void* dst, int pitch, cudaStream_t stream);
int nchw_to_nhwc_tf32(const float* src, int N, int C, int hw, float* dst, int pitch, cudaStream_t stream);   // fp32 NHWC, TF32-rounded
int seam_tail_backward(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc, float* didentity,
                       cudaStream_t stream);
int seam_conv3_g(const void* dy, const void* y, int N, int C, int hw, void* g, float* didentity, cudaStream_t stream);
long long bn_stats_scratch_bytes(int N, int C);
int bn_stats(const float* c, int N, int C, int hw, void* scratch, long long scratch_bytes, double* record, cudaStream_t stream);
int bn_combine_stats(const double* records, int R, int C, float eps, float momentum, const long long* num_batches_tracked,
                     float* running_mean, float* running_var, float* mean, float* invstd, double* count, cudaStream_t stream);
int seam_tail_bn_forward(const float* c, const float* identity, const float* mean, const float* invstd, const float* gamma,
                         const float* beta, int N, int C, int hw, void* y, cudaStream_t stream);
long long seam_tail_bn_backward_reduce_scratch_bytes(int N, int C, int hw);
int seam_tail_bn_backward_reduce(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, int N, int C,
                                 int hw, void* scratch, long long scratch_bytes, float* sums, float* dgamma, float* dbeta,
                                 cudaStream_t stream);
int seam_tail_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                          const float* sums, int R, const double* count, int N, int C, int hw, float* dc, float* didentity,
                          cudaStream_t stream);
int seam_tail_bn_backward_g(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                            const float* sums, int R, const double* count, int N, int C, int hw, void* g, float* didentity,
                            cudaStream_t stream);

// ---- seam_conv3.cu ----
long long seam_conv3_workspace_bytes(int N, int Cin, int Cout, int hw);
int seam_conv3_forward(const float* out2, const float* identity, const float* w3, const float* scale, const float* bias, int N, int Cin,
                       int Cout, int hw, void* ws, long long ws_bytes, void* y, cudaStream_t stream);
long long seam_conv3_backward_scratch_bytes(int N, int Cin, int Cout, int hw);
int seam_conv3_backward(const void* dy, const void* y, const void* ws, const float* scale, int N, int Cin, int Cout, int hw,
                        void* scratch, long long scratch_bytes, float* d_out2, float* dw3, float* didentity, cudaStream_t stream);
long long seam_conv3_bn_forward_scratch_bytes(int N, int Cout, int hw);
long long seam_conv3_bn_backward_scratch_bytes(int N, int Cin, int Cout, int hw);
int seam_conv3_bn_forward(const float* out2, const float* w3, int N, int Cin, int Cout, int hw, void* ws, long long ws_bytes,
                          void* scratch, long long scratch_bytes, float* c, double* record, cudaStream_t stream);
int seam_conv3_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                           const float* sums, int R, const double* count, const void* ws, int N, int Cin, int Cout, int hw,
                           void* scratch, long long scratch_bytes, float* d_out2, float* dw3, float* didentity, cudaStream_t stream);

// ---- tta_kernels.cu ----
int tta_launch(const float* const* logits, const int* hs, const int* ws, const int* flips, int n_maps, int C, const void* labels,
               int label_bytes, int H, int W, int ignore_index, const float* divisors, int n_div, int div_exact, long long* cm,
               void* pred, int pred_bytes, float* probs, cudaStream_t stream);
void tta_set_row_walk(int on);

// ---- optim_kernels.cu ----
int sgd_step(int n_tensors, float* const* params, const float* const* grads, float* const* momentum_bufs, const long long* numels,
             float lr, float momentum, float dampening, float weight_decay, int nesterov, int first_step, float grad_scale,
             cudaStream_t stream);
int adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
              const long long* numels, float lr, float beta1, float beta2, float eps, float weight_decay, long long step,
              float grad_scale, cudaStream_t stream);

// ---- p2p_allreduce.cu ----
int p2p_allreduce_mean(void* const* peer_bufs, void* multicast_ptr, void* const* signal_pads, int rank, int world, long long numel,
                       int blocks, int pad_slot0, cudaStream_t stream);

}  // namespace b200seg
