// extern "C" boundary of libb200seg.so (declarations + reference citations: include/b200seg.h)
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include "../../include/b200seg.h"
#include "common.cuh"

namespace b200seg {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static long long g_launches = 0;
void count_launch() { __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED); }

// ---- optional per-kernel event timing (bench.py roofline leg) ---------------------------------
constexpr int PROF_TAGS = 16, PROF_MAX = 4096;
static int g_prof_on = 0;
static int g_prof_n[PROF_TAGS];
static cudaEvent_t g_prof_ev[PROF_TAGS][PROF_MAX][2];
void profile_begin(int tag, cudaStream_t stream) {
  if (!g_prof_on || tag < 0 || tag >= PROF_TAGS || g_prof_n[tag] >= PROF_MAX) return;
  cudaEvent_t* e = g_prof_ev[tag][g_prof_n[tag]];
  cudaEventCreate(&e[0]); cudaEventCreate(&e[1]);
  cudaEventRecord(e[0], stream);
}
void profile_end(int tag, cudaStream_t stream) {
  if (!g_prof_on || tag < 0 || tag >= PROF_TAGS || g_prof_n[tag] >= PROF_MAX) return;
  cudaEventRecord(g_prof_ev[tag][g_prof_n[tag]][1], stream);
  ++g_prof_n[tag];
}

int num_sms() {
  static int cached = 0;
  if (cached <= 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// kernels' host launchers (defined in the other translation units)
int k4_launch(const float*, int, int, int, int, const void*, int, int, int, int, long long*, long long, void*, int, int, cudaStream_t);
int k4_launch_frames(const float* const*, int, int, int, int, const void* const*, int, int, int, int, long long*, long long, void* const*,
                     int, int, cudaStream_t);
int confusion_pairs_launch_ex(void*, int, const void*, int, long long, int, int, int, long long*, cudaStream_t);
long long k2_workspace_bytes(int, int, int, int, int, int);
int k2_forward(const float*, int, int, int, int, const void*, int, int, int, int, float, int, void*, long long, float*, cudaStream_t,
               float* loss_copy = nullptr);
int k2_backward_packed_multi(void*, int, int, int, int, int, int, float, const float*, const float*, void*, float* const*, int, cudaStream_t);
void* aspp_bwd_gOt_ptr(void*);
int k2_backward(const void*, int, int, int, int, int, int, float, const float*, const float*, float*, cudaStream_t);
int k2_backward_packed(void*, int, int, int, int, int, int, float, const float*, const float*, void*, float*, cudaStream_t);
int aspp_backward_packed(const void*, const void*, const void*, const int*, int, int, int, int, int, int, void*, long long, int, float*,
                         float* const*, cudaStream_t, void*, cudaEvent_t);
int upsample_fwd_launch(const float*, float*, int, int, int, int, int, int, cudaStream_t);
int upsample_bwd_launch(const float*, float*, int, int, int, int, int, cudaStream_t);
long long k3_workspace_bytes();
long long k3_stats_bytes(int, int, int);
int k3_forward(const float*, const float*, const float*, int, int, int, int, void*, long long, float*, cudaStream_t, float*);
int k3_backward(const float*, const float*, const float*, const float*, int, int, int, int, float*, cudaStream_t, const float*);
int aspp_nj(int, int);
int aspp_pack_weights(const float* const*, const float* const*, int, int, int, void*, void*, float*, cudaStream_t);
int aspp_pack_features(const float*, int, int, int, int, void*, cudaStream_t);
long long aspp_yt_bytes(int, int, int, int, int);
int aspp_forward(const void*, const void*, const float*, const int*, int, int, int, int, int, int, float*, float*, cudaStream_t);
int aspp_forward_f32(const float*, const void*, const float*, const int*, int, int, int, int, int, int, float*, float*, void*, cudaStream_t);
int aspp_forward_f32_supported(const float*, int, int, int, int, int);
long long aspp_bwd_scratch_bytes(int, int, int, int, int, int, int);
int aspp_backward(const float*, const void*, const void*, const int*, int, int, int, int, int, int, void*, long long, int, float*,
                  float* const*, float* const*, cudaStream_t);
long long k5_workspace_bytes(int, int, int, int, int, int);
int k5_forward(const float*, const float*, int, int, int, int, int, int, float, float, int, int, void*, long long, float*, cudaStream_t);
int k5_backward(const void*, int, int, int, int, int, int, const float*, const float*, float*, cudaStream_t);
int conv3x3_pack_weights(const float* const*, const int*, int, int, void*, void*, int, cudaStream_t);
int conv3x3_pack_weights_stack(int, const float* const*, const int*, const int*, const int*, void* const*, void* const*, const int*,
                               const float* const*, const int*, int, float*, cudaStream_t);
int conv3x3_forward(const void*, int, int, int, int, long long, const void*, int, int, const float*, int, float, void*, long long, float*,
                    cudaStream_t);
int conv3x3_dgrad(const void*, int, int, int, int, long long, const void*, int, int, const void*, float, void*, long long, float*,
                  cudaStream_t, void*, long long, float*);
long long conv3x3_dgrad_colsum_scratch_bytes(int, int, int, long long);
long long conv3x3_wgrad_scratch_bytes(int, int, int, int, int, int);
int conv3x3_wgrad(const void*, int, long long, const void*, int, long long, int, int, int, int, int, void*, long long, float* const*,
                  const int*, int, cudaStream_t);
int nchw_to_nhwc_bf16(const float*, int, int, int, void*, int, cudaStream_t);
int seam_tail_forward(const float*, const float*, const float*, const float*, int, int, int, void*, cudaStream_t);
int seam_tail_backward(const void*, const void*, const float*, int, int, int, float*, float*, cudaStream_t);
long long seam_conv3_workspace_bytes(int, int, int, int);
int seam_conv3_forward(const float*, const float*, const float*, const float*, const float*, int, int, int, int, void*, long long, void*,
                       cudaStream_t);
long long seam_conv3_backward_scratch_bytes(int, int, int, int);
int seam_conv3_backward(const void*, const void*, const void*, const float*, int, int, int, int, void*, long long, float*, float*, float*,
                        cudaStream_t);
long long bn_stats_scratch_bytes(int, int);
int bn_stats(const float*, int, int, int, void*, long long, double*, cudaStream_t);
int bn_combine_stats(const double*, int, int, float, float, const long long*, float*, float*, float*, float*, double*, cudaStream_t);
int seam_tail_bn_forward(const float*, const float*, const float*, const float*, const float*, const float*, int, int, int, void*,
                         cudaStream_t);
long long seam_tail_bn_backward_reduce_scratch_bytes(int, int, int);
int seam_tail_bn_backward_reduce(const void*, const void*, const float*, const float*, const float*, int, int, int, void*, long long,
                                 float*, float*, float*, cudaStream_t);
int seam_tail_bn_backward(const void*, const void*, const float*, const float*, const float*, const float*, const float*, int,
                          const double*, int, int, int, float*, float*, cudaStream_t);
long long seam_conv3_bn_forward_scratch_bytes(int, int, int);
long long seam_conv3_bn_backward_scratch_bytes(int, int, int, int);
int seam_conv3_bn_forward(const float*, const float*, int, int, int, int, void*, long long, void*, long long, float*, double*, cudaStream_t);
int seam_conv3_bn_backward(const void*, const void*, const float*, const float*, const float*, const float*, const float*, int,
                           const double*, const void*, int, int, int, int, void*, long long, float*, float*, float*, cudaStream_t);
long long nhwc_colsum_scratch_bytes(int);
int nhwc_bf16_colsum(const void*, long long, int, int, void*, float*, cudaStream_t);
int tta_launch(const float* const*, const int*, const int*, const int*, int, int, const void*, int, int, int, int, const float*, int, int,
               long long*, void*, int, float*, cudaStream_t);
void tta_set_row_walk(int);
void k2_set_variant(int);
int p2p_allreduce_mean(void* const*, void*, void* const*, int, int, long long, int, int, cudaStream_t);
int sgd_step(int, float* const*, const float* const*, float* const*, const long long*, float, float, float, float, int, int, float,
             cudaStream_t);
int adam_step(int, float* const*, const float* const*, float* const*, float* const*, const long long*, float, float, float, float,
              float, long long, float, cudaStream_t);
namespace gemm { namespace conv { void set_pair(int); } }
namespace gemm {
int selftest(int, int, int, int, int, int, int, int, double*, double*);
void set_sharing(int);
void set_overlap_sms(int);
void set_narrow_tiles(int);
void set_dgrad_mode(int);
void set_fwd_mode(int);
void set_fwd_convert(int);
int selftest_fwd_convert(int, int, int, int, int, double*, double*, double*);
}

static int require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    set_error("no CUDA device available (%s); b200seg has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return B200SEG_ERR_CUDA;
  }
  return B200SEG_OK;
}

}  // namespace b200seg

using namespace b200seg;
#define S(stream) reinterpret_cast<cudaStream_t>(stream)

// ---------------------------------------------------------------------------------------------------------------------------
// Replay of the one-call train entries from CUDA graphs.  The sequence a call enqueues is a pure function of its arguments
// (pointers, shapes, scalars) and of the library's global switches, so the second time the SAME arguments are seen the sequence
// is captured on a private stream and from then on replayed with one cudaGraphLaunch on the caller's stream -- a training loop
// in steady state hands the same addresses back every iteration (caching allocator), and ~7 launches per direction become one.
// Anything that makes the replay unsafe or pointless takes the direct path: caller already capturing, per-kernel profiling on,
// a switch flipped (all graphs dropped), addresses that keep changing (cache turns itself off).
// ---------------------------------------------------------------------------------------------------------------------------
struct StepKey {
  const void* p[28];
  long long i[24];
  float f[4];
};
struct StepGraph {
  StepKey key;
  cudaGraphExec_t exec;
  long long launches;
  unsigned long long stamp;
  bool used;
};
constexpr int STEP_GRAPHS = 16;
static StepGraph g_step_graphs[STEP_GRAPHS];
static cudaStream_t g_step_capture_stream[64];
static int g_step_graphs_on = -1;                 // -1: read B200SEG_STEP_GRAPHS on first use
static long long g_step_hits = 0, g_step_captures = 0;
static unsigned long long g_step_stamp = 0;
static int g_step_lock = 0;
struct StepLock {
  StepLock() { while (__atomic_exchange_n(&g_step_lock, 1, __ATOMIC_ACQUIRE)) {} }
  ~StepLock() { __atomic_store_n(&g_step_lock, 0, __ATOMIC_RELEASE); }
};

static void step_graphs_drop_locked() {
  for (int q = 0; q < STEP_GRAPHS; ++q) {
    if (g_step_graphs[q].exec) cudaGraphExecDestroy(g_step_graphs[q].exec);
    g_step_graphs[q] = StepGraph{};
  }
}
static void step_graphs_drop() {
  StepLock lock;
  step_graphs_drop_locked();
}

template <class Body>
static int run_step(const StepKey& key, cudaStream_t stream, bool allow_graph, Body&& body) {
  if (g_step_graphs_on < 0) {
    const char* e = getenv("B200SEG_STEP_GRAPHS");
    g_step_graphs_on = (e && e[0] == '0') ? 0 : 1;
  }
  if (!allow_graph || !g_step_graphs_on || g_prof_on) return body(stream);
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) {
    cudaGetLastError();
    return body(stream);
  }
  StepLock lock;
  int slot = -1, lru = 0;                                                        // lru: a free slot, else the least recently used
  for (int q = 0; q < STEP_GRAPHS; ++q) {
    const StepGraph& c = g_step_graphs[q];
    if (c.used && memcmp(&c.key, &key, sizeof(StepKey)) == 0) { slot = q; break; }
    const StepGraph& b = g_step_graphs[lru];
    if ((!c.used && b.used) || (c.used == b.used && c.stamp < b.stamp)) lru = q;
  }
  if (slot >= 0 && g_step_graphs[slot].exec) {                                   // replay
    StepGraph& g = g_step_graphs[slot];
    g.stamp = ++g_step_stamp;
    ++g_step_hits;
    __atomic_add_fetch(&g_launches, g.launches, __ATOMIC_RELAXED);
    B200SEG_CUDA(cudaGraphLaunch(g.exec, stream));
    return B200SEG_OK;
  }
  if (slot < 0) {                                                                // first sight: remember, run directly
    StepGraph& g = g_step_graphs[lru];
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g = StepGraph{};
    g.key = key; g.used = true; g.stamp = ++g_step_stamp;
    return body(stream);
  }
  // second sight: capture on the private stream, instantiate, launch on the caller's stream
  if (g_step_captures >= 48 && g_step_hits < 2 * g_step_captures) {             // addresses keep changing: stop trying
    g_step_graphs_on = 0;
    step_graphs_drop_locked();
    return body(stream);
  }
  int dev = 0;
  B200SEG_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return body(stream);
  if (!g_step_capture_stream[dev]) B200SEG_CUDA(cudaStreamCreateWithFlags(&g_step_capture_stream[dev], cudaStreamNonBlocking));
  cudaStream_t cs = g_step_capture_stream[dev];
  if (cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
    cudaGetLastError();
    return body(stream);
  }
  const long long l0 = g_launches;
  const int rc = body(cs);
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(cs, &graph);
  const long long captured = g_launches - l0;
  __atomic_sub_fetch(&g_launches, captured, __ATOMIC_RELAXED);                   // nothing has run yet
  if (rc != B200SEG_OK || e != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    g_step_graphs[slot] = StepGraph{};
    return rc != B200SEG_OK ? rc : body(stream);
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t e2 = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess || !exec) {
    cudaGetLastError();
    g_step_graphs[slot] = StepGraph{};
    return body(stream);
  }
  StepGraph& g = g_step_graphs[slot];
  g.exec = exec; g.launches = captured; g.stamp = ++g_step_stamp;
  ++g_step_captures;
  __atomic_add_fetch(&g_launches, captured, __ATOMIC_RELAXED);
  B200SEG_CUDA(cudaGraphLaunch(exec, stream));
  return B200SEG_OK;
}
#define REQUIRE_DEVICE()                 \
  do {                                   \
    int rc__ = require_device();         \
    if (rc__) return rc__;               \
  } while (0)

extern "C" {

int b200seg_abi_version(void) { return B200SEG_ABI_VERSION; }
const char* b200seg_last_error(void) { return g_err; }
int b200seg_device_sms(void) {
  if (require_device()) return -1;
  return num_sms();
}

int b200seg_upsample_argmax_confusion(const float* logits, int N, int C, int h, int w, const int64_t* labels, int H, int W,
                                      int ignore_index, int64_t* cm, int64_t cm_frame_stride, int64_t* pred, int fma_mode,
                                      void* stream) {
  REQUIRE_DEVICE();
  return k4_launch(logits, N, C, h, w, labels, 8, H, W, ignore_index, reinterpret_cast<long long*>(cm), cm_frame_stride, pred, 8,
                   fma_mode, S(stream));
}

int b200seg_upsample_argmax_confusion_ex(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H,
                                         int W, int ignore_index, int64_t* cm, int64_t cm_frame_stride, void* pred, int pred_bytes,
                                         int fma_mode, void* stream) {
  REQUIRE_DEVICE();
  return k4_launch(logits, N, C, h, w, labels, label_bytes, H, W, ignore_index, reinterpret_cast<long long*>(cm), cm_frame_stride,
                   pred, pred_bytes, fma_mode, S(stream));
}

int b200seg_upsample_argmax_confusion_frames(const float* const* logits_host, int n_frames, int C, int h, int w,
                                             const void* const* labels_host, int label_bytes, int H, int W, int ignore_index,
                                             int64_t* cm, int64_t cm_frame_stride, void* const* pred_host, int pred_bytes,
                                             void* stream) {
  REQUIRE_DEVICE();
  return k4_launch_frames(logits_host, n_frames, C, h, w, labels_host, label_bytes, H, W, ignore_index,
                          reinterpret_cast<long long*>(cm), cm_frame_stride, pred_host, pred_bytes, 0, S(stream));
}

int b200seg_confusion_from_pred(int64_t* pd, const int64_t* gt, int64_t n, int C, int ignore_index, int mutate_pd, int64_t* cm,
                                void* stream) {
  REQUIRE_DEVICE();
  return confusion_pairs_launch_ex(pd, 8, gt, 8, n, C, ignore_index, mutate_pd, reinterpret_cast<long long*>(cm), S(stream));
}

int b200seg_confusion_from_pred_ex(void* pd, int pd_bytes, const void* gt, int gt_bytes, int64_t n, int C, int ignore_index,
                                   int mutate_pd, int64_t* cm, void* stream) {
  REQUIRE_DEVICE();
  return confusion_pairs_launch_ex(pd, pd_bytes, gt, gt_bytes, n, C, ignore_index, mutate_pd, reinterpret_cast<long long*>(cm), S(stream));
}

int64_t b200seg_upsample_ce_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  if (N <= 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
  return k2_workspace_bytes(N, C, h, w, H, W);
}

int b200seg_upsample_ce_forward(const float* logits, int N, int C, int h, int w, const int64_t* labels, int H, int W,
                                int ignore_index, float inv_temperature, int need_grad, void* workspace, int64_t workspace_bytes,
                                float* loss_out2, void* stream) {
  REQUIRE_DEVICE();
  return k2_forward(logits, N, C, h, w, labels, 8, H, W, ignore_index, inv_temperature, need_grad, workspace, workspace_bytes,
                    loss_out2, S(stream));
}

int b200seg_upsample_ce_forward_ex(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H, int W,
                                   int ignore_index, float inv_temperature, int need_grad, void* workspace, int64_t workspace_bytes,
                                   float* loss_out2, void* stream) {
  REQUIRE_DEVICE();
  return k2_forward(logits, N, C, h, w, labels, label_bytes, H, W, ignore_index, inv_temperature, need_grad, workspace,
                    workspace_bytes, loss_out2, S(stream));
}

int b200seg_upsample_ce_backward(const void* workspace, int N, int C, int h, int w, int H, int W, float inv_temperature,
                                 const float* loss_out2, const float* grad_out, float* grad_logits, void* stream) {
  REQUIRE_DEVICE();
  return k2_backward(workspace, N, C, h, w, H, W, inv_temperature, loss_out2, grad_out, grad_logits, S(stream));
}

int b200seg_upsample_ce_backward_packed(void* workspace, int N, int C, int h, int w, int H, int W, float inv_temperature,
                                        const float* loss_out2, const float* grad_out, void* gOt, float* bias_grad, void* stream) {
  REQUIRE_DEVICE();
  return k2_backward_packed(workspace, N, C, h, w, H, W, inv_temperature, loss_out2, grad_out, gOt, bias_grad, S(stream));
}

int b200seg_aspp_backward_packed(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N, int Cin, int C,
                                 int h, int w, void* scratch, int64_t scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                                 void* stream) {
  REQUIRE_DEVICE();
  return aspp_backward_packed(gOt, Xp, WpT, rates_host, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, grad_x, grad_w, S(stream),
                              nullptr, nullptr);
}

int b200seg_aspp_backward_packed_nhwc(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N, int Cin,
                                      int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits, void* grad_x_nhwc_bf16,
                                      float* const* grad_w, void* stream) {
  REQUIRE_DEVICE();
  return aspp_backward_packed(gOt, Xp, WpT, rates_host, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, nullptr, grad_w, S(stream),
                              grad_x_nhwc_bf16, nullptr);
}

int b200seg_aspp_backward_packed_ex(const void* gOt, const void* Xp, const void* WpT, const int* rates_host, int R, int N, int Cin,
                                    int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits, float* grad_x,
                                    void* grad_x_nhwc_bf16, float* const* grad_w, void* weights_ready_event, void* stream) {
  REQUIRE_DEVICE();
  return aspp_backward_packed(gOt, Xp, WpT, rates_host, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, grad_x, grad_w, S(stream),
                              grad_x_nhwc_bf16, reinterpret_cast<cudaEvent_t>(weights_ready_event));
}

int b200seg_upsample_bilinear_forward(const float* in, float* out, int NC, int h, int w, int H, int W, int fma_mode, void* stream) {
  REQUIRE_DEVICE();
  return upsample_fwd_launch(in, out, NC, h, w, H, W, fma_mode, S(stream));
}

int b200seg_upsample_bilinear_backward(const float* grad_out, float* grad_in, int NC, int h, int w, int H, int W, void* stream) {
  REQUIRE_DEVICE();
  return upsample_bwd_launch(grad_out, grad_in, NC, h, w, H, W, S(stream));
}

int64_t b200seg_soft_ce_workspace_bytes(void) { return k3_workspace_bytes(); }

int b200seg_soft_ce_forward(const float* pred, const float* soft, const float* weights, int N, int K, int H, int W, void* workspace,
                            int64_t workspace_bytes, float* loss_out, void* stream) {
  REQUIRE_DEVICE();
  return k3_forward(pred, soft, weights, N, K, H, W, workspace, workspace_bytes, loss_out, S(stream), nullptr);
}

int b200seg_soft_ce_backward(const float* pred, const float* soft, const float* weights, const float* grad_out, int N, int K, int H,
                             int W, float* grad_pred, void* stream) {
  REQUIRE_DEVICE();
  return k3_backward(pred, soft, weights, grad_out, N, K, H, W, grad_pred, S(stream), nullptr);
}

int64_t b200seg_soft_ce_stats_bytes(int N, int H, int W) { return k3_stats_bytes(N, H, W); }

int b200seg_soft_ce_forward_stats(const float* pred, const float* soft, const float* weights, int N, int K, int H, int W,
                                  void* workspace, int64_t workspace_bytes, float* stats, float* loss_out, void* stream) {
  REQUIRE_DEVICE();
  return k3_forward(pred, soft, weights, N, K, H, W, workspace, workspace_bytes, loss_out, S(stream), stats);
}

int b200seg_soft_ce_backward_stats(const float* pred, const float* soft, const float* weights, const float* stats,
                                   const float* grad_out, int N, int K, int H, int W, float* grad_pred, void* stream) {
  REQUIRE_DEVICE();
  B200SEG_CHECK_ARG(stats != nullptr, "soft_ce_backward_stats: stats is null");
  return k3_backward(pred, soft, weights, grad_out, N, K, H, W, grad_pred, S(stream), stats);
}

int64_t b200seg_fada_softce_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  if (N <= 0 || C <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return 0;
  return k5_workspace_bytes(N, C, h, w, H, W);
}

int b200seg_fada_softce_forward(const float* d_logits, const float* seg_logits, int N, int C, int h, int w, int H, int W,
                                float inv_temperature, float clamp, int slot, int need_grad, void* workspace, int64_t workspace_bytes,
                                float* loss_out2, void* stream) {
  REQUIRE_DEVICE();
  return k5_forward(d_logits, seg_logits, N, C, h, w, H, W, inv_temperature, clamp, slot, need_grad, workspace, workspace_bytes,
                    loss_out2, S(stream));
}

int b200seg_fada_softce_backward(const void* workspace, int N, int C, int h, int w, int H, int W, const float* loss_out2,
                                 const float* grad_out, float* grad_d_logits, void* stream) {
  REQUIRE_DEVICE();
  return k5_backward(workspace, N, C, h, w, H, W, loss_out2, grad_out, grad_d_logits, S(stream));
}

int b200seg_aspp_packed_rows(int C, int R) { return aspp_nj(C, R); }

int b200seg_aspp_pack_weights(const float* const* weights, const float* const* biases, int R, int C, int Cin, void* Wp, void* WpT,
                              float* bias_sum, void* stream) {
  REQUIRE_DEVICE();
  return aspp_pack_weights(weights, biases, R, C, Cin, Wp, WpT, bias_sum, S(stream));
}

int b200seg_aspp_pack_features(const float* x_nchw, int N, int Cin, int h, int w, void* Xp, void* stream) {
  REQUIRE_DEVICE();
  return aspp_pack_features(x_nchw, N, Cin, h, w, Xp, S(stream));
}

int64_t b200seg_aspp_forward_scratch_bytes(int N, int C, int h, int w, int R) {
  if (N <= 0 || C <= 0 || h <= 0 || w <= 0 || R <= 0) return 0;
  return aspp_yt_bytes(N, C, h, w, R);
}

int b200seg_aspp_forward(const void* Xp, const void* Wp, const float* bias_sum, const int* rates_host, int R, int N, int Cin, int C,
                         int h, int w, void* scratch, float* logits, void* stream) {
  REQUIRE_DEVICE();
  return aspp_forward(Xp, Wp, bias_sum, rates_host, R, N, Cin, C, h, w, reinterpret_cast<float*>(scratch), logits, S(stream));
}

int b200seg_aspp_forward_f32_supported(const float* x, int Cin, int C, int h, int w, int R) {
  return aspp_forward_f32_supported(x, Cin, C, h, w, R);
}

int b200seg_aspp_forward_f32(const float* x, const void* Wp, const float* bias_sum, const int* rates_host, int R, int N, int Cin, int C,
                             int h, int w, void* scratch, float* logits, void* xn_bf16_nchw, void* stream) {
  REQUIRE_DEVICE();
  return aspp_forward_f32(x, Wp, bias_sum, rates_host, R, N, Cin, C, h, w, reinterpret_cast<float*>(scratch), logits, xn_bf16_nchw, S(stream));
}

int64_t b200seg_aspp_backward_scratch_bytes(int N, int Cin, int C, int h, int w, int R, int splits) {
  if (N <= 0 || C <= 0 || h <= 0 || w <= 0 || R <= 0) return 0;
  return aspp_bwd_scratch_bytes(N, Cin, C, h, w, R, splits < 1 ? 1 : splits);
}

int b200seg_aspp_backward(const float* grad_logits, const void* Xp, const void* WpT, const int* rates_host, int R, int N, int Cin,
                          int C, int h, int w, void* scratch, int64_t scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                          float* const* grad_b, void* stream) {
  REQUIRE_DEVICE();
  return aspp_backward(grad_logits, Xp, WpT, rates_host, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, grad_x, grad_w, grad_b,
                       S(stream));
}

int b200seg_conv3x3_pack_weights(const float* const* weights, const int* part_co_host, int n_parts, int Ci, void* Wf, void* Wb,
                                 int co_pitch, void* stream) {
  REQUIRE_DEVICE();
  return conv3x3_pack_weights(weights, part_co_host, n_parts, Ci, Wf, Wb, co_pitch, S(stream));
}

int b200seg_conv3x3_pack_weights_stack(int n_layers, const float* const* weights, const int* part_co_host, const int* parts_per_layer_host,
                                       const int* Ci_host, void* const* Wf, void* const* Wb, const int* co_pitch_host,
                                       const float* const* bias_parts, const int* bias_len_host, int n_bias, float* bias_out,
                                       void* stream) {
  REQUIRE_DEVICE();
  return conv3x3_pack_weights_stack(n_layers, weights, part_co_host, parts_per_layer_host, Ci_host, Wf, Wb, co_pitch_host, bias_parts,
                                    bias_len_host, n_bias, bias_out, S(stream));
}

int b200seg_conv3x3_forward(const void* act, int N, int h, int w, int Ci, int64_t act_pitch, const void* Wf, int Co, int dilation,
                            const float* bias, int lrelu, float slope, void* out_bf16_nhwc, int64_t out_pitch, float* out_f32_nchw,
                            void* stream) {
  REQUIRE_DEVICE();
  return conv3x3_forward(act, N, h, w, Ci, act_pitch, Wf, Co, dilation, bias, lrelu, slope, out_bf16_nhwc, out_pitch, out_f32_nchw,
                         S(stream));
}

int b200seg_conv3x3_dgrad(const void* g, int N, int h, int w, int Cg, int64_t g_pitch, const void* Wb, int Ci, int dilation,
                          const void* mask, float slope, void* out_bf16_nhwc, int64_t out_pitch, float* out_f32_nchw, void* stream) {
  REQUIRE_DEVICE();
  return conv3x3_dgrad(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, mask, slope, out_bf16_nhwc, out_pitch, out_f32_nchw, S(stream),
                       nullptr, 0, nullptr);
}

int64_t b200seg_conv3x3_dgrad_colsum_scratch_bytes(int N, int h, int w, int64_t out_pitch) {
  if (N <= 0 || h <= 0 || w <= 0 || out_pitch <= 0) return 0;
  return conv3x3_dgrad_colsum_scratch_bytes(N, h, w, out_pitch);
}

int b200seg_conv3x3_dgrad_colsum(const void* g, int N, int h, int w, int Cg, int64_t g_pitch, const void* Wb, int Ci, int dilation,
                                 const void* mask, float slope, void* out_bf16_nhwc, int64_t out_pitch, void* colsum_scratch,
                                 int64_t colsum_scratch_bytes, float* colsum_out, void* stream) {
  REQUIRE_DEVICE();
  if (!colsum_out) { set_error("b200seg_conv3x3_dgrad_colsum: colsum_out is null"); return B200SEG_ERR_ARG; }
  return conv3x3_dgrad(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, mask, slope, out_bf16_nhwc, out_pitch, nullptr, S(stream),
                       colsum_scratch, colsum_scratch_bytes, colsum_out);
}

int64_t b200seg_conv3x3_wgrad_scratch_bytes(int N, int h, int w, int Co, int Ci, int splits) {
  if (N <= 0 || h <= 0 || w <= 0 || Co <= 0 || Ci <= 0) return 0;
  return conv3x3_wgrad_scratch_bytes(N, h, w, Co, Ci, splits);
}

int b200seg_conv3x3_wgrad(const void* g, int Co, int64_t g_pitch, const void* x, int Ci, int64_t x_pitch, int N, int h, int w,
                          int dilation, int splits, void* scratch, int64_t scratch_bytes, float* const* grad_w,
                          const int* part_co_host, int n_parts, void* stream) {
  REQUIRE_DEVICE();
  return conv3x3_wgrad(g, Co, g_pitch, x, Ci, x_pitch, N, h, w, dilation, splits, scratch, scratch_bytes, grad_w, part_co_host,
                       n_parts, S(stream));
}

int b200seg_nchw_to_nhwc_bf16(const float* src, int N, int C, int hw, void* dst, int pitch, void* stream) {
  REQUIRE_DEVICE();
  return nchw_to_nhwc_bf16(src, N, C, hw, dst, pitch, S(stream));
}

int b200seg_seam_tail_forward(const float* c, const float* identity, const float* scale, const float* bias, int N, int C, int hw, void* y,
                              void* stream) {
  REQUIRE_DEVICE();
  return seam_tail_forward(c, identity, scale, bias, N, C, hw, y, S(stream));
}

int b200seg_seam_tail_backward(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc, float* didentity,
                               void* stream) {
  REQUIRE_DEVICE();
  return seam_tail_backward(dy, y, scale, N, C, hw, dc, didentity, S(stream));
}

int64_t b200seg_seam_conv3_workspace_bytes(int N, int Cin, int Cout, int hw) { return seam_conv3_workspace_bytes(N, Cin, Cout, hw); }

int b200seg_seam_conv3_forward(const float* out2, const float* identity, const float* w3, const float* scale, const float* bias, int N,
                               int Cin, int Cout, int hw, void* ws, int64_t ws_bytes, void* y, void* stream) {
  REQUIRE_DEVICE();
  return seam_conv3_forward(out2, identity, w3, scale, bias, N, Cin, Cout, hw, ws, ws_bytes, y, S(stream));
}

int64_t b200seg_seam_conv3_backward_scratch_bytes(int N, int Cin, int Cout, int hw) {
  return seam_conv3_backward_scratch_bytes(N, Cin, Cout, hw);
}

int b200seg_seam_conv3_backward(const void* dy, const void* y, const void* ws, const float* scale, int N, int Cin, int Cout, int hw,
                                void* scratch, int64_t scratch_bytes, float* d_out2, float* dw3, float* didentity, void* stream) {
  REQUIRE_DEVICE();
  return seam_conv3_backward(dy, y, ws, scale, N, Cin, Cout, hw, scratch, scratch_bytes, d_out2, dw3, didentity, S(stream));
}

int64_t b200seg_bn_stats_scratch_bytes(int N, int C) { return bn_stats_scratch_bytes(N, C); }

int b200seg_bn_stats(const float* c, int N, int C, int hw, void* scratch, int64_t scratch_bytes, double* record, void* stream) {
  REQUIRE_DEVICE();
  return bn_stats(c, N, C, hw, scratch, scratch_bytes, record, S(stream));
}

int b200seg_bn_combine_stats(const double* records, int R, int C, float eps, float momentum, const int64_t* num_batches_tracked,
                             float* running_mean, float* running_var, float* mean, float* invstd, double* count, void* stream) {
  REQUIRE_DEVICE();
  return bn_combine_stats(records, R, C, eps, momentum, reinterpret_cast<const long long*>(num_batches_tracked), running_mean,
                          running_var, mean, invstd, count, S(stream));
}

int b200seg_seam_tail_bn_forward(const float* c, const float* identity, const float* mean, const float* invstd, const float* gamma,
                                 const float* beta, int N, int C, int hw, void* y, void* stream) {
  REQUIRE_DEVICE();
  return seam_tail_bn_forward(c, identity, mean, invstd, gamma, beta, N, C, hw, y, S(stream));
}

int64_t b200seg_seam_tail_bn_backward_reduce_scratch_bytes(int N, int C, int hw) {
  return seam_tail_bn_backward_reduce_scratch_bytes(N, C, hw);
}

int b200seg_seam_tail_bn_backward_reduce(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, int N,
                                         int C, int hw, void* scratch, int64_t scratch_bytes, float* sums, float* dgamma, float* dbeta,
                                         void* stream) {
  REQUIRE_DEVICE();
  return seam_tail_bn_backward_reduce(dy, y, c, mean, invstd, N, C, hw, scratch, scratch_bytes, sums, dgamma, dbeta, S(stream));
}

int b200seg_seam_tail_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd,
                                  const float* gamma, const float* sums, int R, const double* count, int N, int C, int hw, float* dc,
                                  float* didentity, void* stream) {
  REQUIRE_DEVICE();
  return seam_tail_bn_backward(dy, y, c, mean, invstd, gamma, sums, R, count, N, C, hw, dc, didentity, S(stream));
}

// conv3 under batch statistics (resnet.py:106-113): the workspace has the fused conv3's layout
int64_t b200seg_seam_conv3_bn_workspace_bytes(int N, int Cin, int Cout, int hw) { return seam_conv3_workspace_bytes(N, Cin, Cout, hw); }

int64_t b200seg_seam_conv3_bn_forward_scratch_bytes(int N, int Cout, int hw) { return seam_conv3_bn_forward_scratch_bytes(N, Cout, hw); }

int b200seg_seam_conv3_bn_forward(const float* out2, const float* w3, int N, int Cin, int Cout, int hw, void* ws, int64_t ws_bytes,
                                  void* scratch, int64_t scratch_bytes, float* c, double* record, void* stream) {
  REQUIRE_DEVICE();
  return seam_conv3_bn_forward(out2, w3, N, Cin, Cout, hw, ws, ws_bytes, scratch, scratch_bytes, c, record, S(stream));
}

int64_t b200seg_seam_conv3_bn_backward_scratch_bytes(int N, int Cin, int Cout, int hw) {
  return seam_conv3_bn_backward_scratch_bytes(N, Cin, Cout, hw);
}

int b200seg_seam_conv3_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd,
                                   const float* gamma, const float* sums, int R, const double* count, const void* ws, int N, int Cin,
                                   int Cout, int hw, void* scratch, int64_t scratch_bytes, float* d_out2, float* dw3, float* didentity,
                                   void* stream) {
  REQUIRE_DEVICE();
  return seam_conv3_bn_backward(dy, y, c, mean, invstd, gamma, sums, R, count, ws, N, Cin, Cout, hw, scratch, scratch_bytes, d_out2, dw3,
                                didentity, S(stream));
}

int b200seg_tta_argmax_confusion(const float* const* logits_lr, const int* h, const int* w, const int* flip, int n_members, int C,
                                 const int64_t* labels, int H, int W, int ignore_index, const float* divisors, int n_div,
                                 int div_exact, int64_t* cm, int64_t* pred, float* probs, void* stream) {
  REQUIRE_DEVICE();
  return tta_launch(logits_lr, h, w, flip, n_members, C, labels, 8, H, W, ignore_index, divisors, n_div, div_exact,
                    reinterpret_cast<long long*>(cm), pred, 8, probs, S(stream));
}

int b200seg_tta_argmax_confusion_ex(const float* const* logits_lr, const int* h, const int* w, const int* flip, int n_members, int C,
                                    const void* labels, int label_bytes, int H, int W, int ignore_index, const float* divisors,
                                    int n_div, int div_exact, int64_t* cm, void* pred, int pred_bytes, float* probs, void* stream) {
  REQUIRE_DEVICE();
  return tta_launch(logits_lr, h, w, flip, n_members, C, labels, label_bytes, H, W, ignore_index, divisors, n_div, div_exact,
                    reinterpret_cast<long long*>(cm), pred, pred_bytes, probs, S(stream));
}

void b200seg_tta_set_row_walk(int on) { tta_set_row_walk(on); }
void b200seg_upsample_ce_set_variant(int v) { step_graphs_drop(); k2_set_variant(v); }

int b200seg_p2p_allreduce_mean(void* const* peer_bufs_host, void* multicast_ptr, void* const* signal_pads_host, int rank, int world,
                               int64_t numel, int blocks, int pad_slot0, void* stream) {
  REQUIRE_DEVICE();
  return p2p_allreduce_mean(peer_bufs_host, multicast_ptr, signal_pads_host, rank, world, numel, blocks, pad_slot0, S(stream));
}

int b200seg_sgd_step(int n_tensors, float* const* params, const float* const* grads, float* const* momentum_bufs,
                     const int64_t* numels, float lr, float momentum, float dampening, float weight_decay, int nesterov,
                     int first_step, float grad_scale, void* stream) {
  REQUIRE_DEVICE();
  return sgd_step(n_tensors, params, grads, momentum_bufs, reinterpret_cast<const long long*>(numels), lr, momentum, dampening,
                  weight_decay, nesterov, first_step, grad_scale, S(stream));
}

int b200seg_adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                      float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2, float eps,
                      float weight_decay, int64_t step, float grad_scale, void* stream) {
  REQUIRE_DEVICE();
  return adam_step(n_tensors, params, grads, exp_avg, exp_avg_sq, reinterpret_cast<const long long*>(numels), lr, beta1, beta2, eps,
                   weight_decay, step, grad_scale, S(stream));
}

int64_t b200seg_nhwc_colsum_scratch_bytes(int pitch) { return pitch > 0 ? nhwc_colsum_scratch_bytes(pitch) : 0; }

int b200seg_nhwc_bf16_colsum(const void* g, int64_t P, int C, int pitch, void* scratch, float* out, void* stream) {
  REQUIRE_DEVICE();
  return nhwc_bf16_colsum(g, P, C, pitch, scratch, out, S(stream));
}

long long b200seg_launch_count(void) { return g_launches; }

void b200seg_profile_enable(int on) {
  step_graphs_drop();
  for (int t = 0; t < PROF_TAGS; ++t) {
    for (int i = 0; i < g_prof_n[t]; ++i) { cudaEventDestroy(g_prof_ev[t][i][0]); cudaEventDestroy(g_prof_ev[t][i][1]); }
    g_prof_n[t] = 0;
  }
  g_prof_on = on;
}

int b200seg_profile_read(int tag, double* total_ms, int* count) {
  if (tag < 0 || tag >= PROF_TAGS || !total_ms || !count) { set_error("profile_read: bad arguments"); return B200SEG_ERR_ARG; }
  double tot = 0.0;
  for (int i = 0; i < g_prof_n[tag]; ++i) {
    B200SEG_CUDA(cudaEventSynchronize(g_prof_ev[tag][i][1]));
    float ms = 0.f;
    B200SEG_CUDA(cudaEventElapsedTime(&ms, g_prof_ev[tag][i][0], g_prof_ev[tag][i][1]));
    tot += ms;
  }
  *total_ms = tot; *count = g_prof_n[tag];
  return B200SEG_OK;
}

void b200seg_conv_set_pair(int on) { step_graphs_drop(); gemm::conv::set_pair(on); }
void b200seg_gemm_set_sharing(int on) { step_graphs_drop(); gemm::set_sharing(on); }
void b200seg_gemm_set_narrow_tiles(int on) { step_graphs_drop(); gemm::set_narrow_tiles(on); }
void b200seg_gemm_set_dgrad_mode(int mode) { step_graphs_drop(); gemm::set_dgrad_mode(mode); }
void b200seg_gemm_set_fwd_mode(int mode) { step_graphs_drop(); gemm::set_fwd_mode(mode); }
void b200seg_gemm_set_fwd_convert(int on) { step_graphs_drop(); gemm::set_fwd_convert(on); }
int b200seg_gemm_fwd_convert_selftest(int M, int n_img, int hw, int K, int write_xn, double* max_err, double* max_ref, double* xn_err) {
  REQUIRE_DEVICE();
  return gemm::selftest_fwd_convert(M, n_img, hw, K, write_xn, max_err, max_ref, xn_err);
}
void b200seg_gemm_set_overlap_sms(int n) { step_graphs_drop(); gemm::set_overlap_sms(n); }

int b200seg_gemm_selftest(int M, int N, int K, int a_mn_major, int b_mn_major, int splits, int col_hw, int share, double* max_err,
                          double* max_ref) {
  REQUIRE_DEVICE();
  if (!max_err || !max_ref) {
    set_error("gemm_selftest: null output pointer");
    return B200SEG_ERR_ARG;
  }
  return gemm::selftest(M, N, K, a_mn_major, b_mn_major, splits, col_hw, share, max_err, max_ref);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------------
// One call per direction for the fused train slice  loss = CE(interpolate(head(x), size) / T, labels)
// (aspp_trainer.py:86-93 / aspp_fada.py:88-96; the head is classifier.py:26-31).  The host cost of the step is the enqueue of
// ~12 kernels: issuing them from ONE foreign call each way (instead of eight, each with its own output allocations) is what
// keeps the small BASELINE configs (1-2 images per GPU) GPU-bound in eager mode.
// ---------------------------------------------------------------------------------------------------------------------------
struct HeadLossLayout {
  long long out2, WpT, Xp, k2ws, Wp, bias_sum, total;
};
static long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }
static HeadLossLayout head_loss_layout(int N, int Cin, int C, int h, int w, int R, int H, int W, int x_kind) {
  HeadLossLayout L;
  const long long P = (long long)N * h * w, NJ = aspp_nj(C, R);
  long long o = 0;
  L.out2 = o; o += 1024;
  L.bias_sum = o; o += 1024;
  L.WpT = o; o = align_up(o + (long long)Cin * NJ * 2, 1024);
  L.Wp = o; o = align_up(o + NJ * Cin * 2, 1024);
  L.Xp = o; if (x_kind == 0) o = align_up(o + P * Cin * 2, 1024);
  L.k2ws = o; o = align_up(o + k2_workspace_bytes(N, C, h, w, H, W), 1024);
  L.total = o;
  return L;
}

// smallest split-K factor >= 4 of the weight-gradient GEMM that fills whole rounds of the 74 CTA pairs best (the rule of
// _lib.default_wgrad_splits, restated here so the one-call entry needs no host-side planning)
static int head_default_splits(long long P, int C, int Cin, int R) {
  const int NJ = aspp_nj(C, R);
  const long long tiles = (long long)(((NJ + 127) / 128 + 1) / 2) * ((Cin + 255) / 256);
  const long long kb = (P + 63) / 64;
  int best = 1;
  double best_eff = -1.0;
  for (int s = 1; s <= 16 && s <= kb; ++s) {
    const long long units = tiles * s;
    const double eff = (double)units / (double)(((units + 73) / 74) * 74);
    if (s >= 4 && eff > best_eff + 1e-9) { best = s; best_eff = eff; }
  }
  if (best_eff > 0) return best;
  return (int)(kb < 1 ? 1 : (kb < 4 ? kb : 4));
}

extern "C" {

int b200seg_aspp_default_wgrad_splits(int64_t P, int C, int Cin, int R) { return head_default_splits(P, C, Cin, R); }

int64_t b200seg_head_loss_workspace_bytes(int N, int Cin, int C, int h, int w, int R, int H, int W, int x_kind) {
  if (N <= 0 || Cin <= 0 || C <= 0 || h <= 0 || w <= 0 || R <= 0 || H <= 0 || W <= 0) return 0;
  return head_loss_layout(N, Cin, C, h, w, R, H, W, x_kind).total;
}

int64_t b200seg_head_loss_scratch_bytes(int N, int Cin, int C, int h, int w, int R) {
  if (N <= 0 || Cin <= 0 || C <= 0 || h <= 0 || w <= 0 || R <= 0) return 0;
  const long long f = aspp_yt_bytes(N, C, h, w, R);
  const long long b = aspp_bwd_scratch_bytes(N, Cin, C, h, w, R, head_default_splits((long long)N * h * w, C, Cin, R));
  return f > b ? f : b;
}

int b200seg_head_loss_forward(const void* x, int x_kind, const float* const* weights, const float* const* biases, const int* rates_host,
                              int R, int N, int Cin, int C, int h, int w, const void* labels, int label_bytes, int H, int W,
                              int ignore_index, float inv_temperature, int need_grad, void* workspace, int64_t workspace_bytes,
                              void* scratch, int64_t scratch_bytes, float* logits, float* loss_out, void* stream) {
  REQUIRE_DEVICE();
  B200SEG_CHECK_ARG(x && weights && rates_host && labels && workspace && scratch && logits && loss_out, "head_loss_forward: null pointer");
  B200SEG_CHECK_ARG(x_kind == 0 || x_kind == 1, "head_loss_forward: x_kind must be 0 (fp32 NCHW) or 1 (bf16 pixel-major), got %d", x_kind);
  B200SEG_CHECK_ARG(N > 0 && Cin > 0 && C > 0 && h > 0 && w > 0 && R > 0 && H > 0 && W > 0, "head_loss_forward: bad shape");
  const HeadLossLayout L = head_loss_layout(N, Cin, C, h, w, R, H, W, x_kind);
  B200SEG_CHECK_ARG(workspace_bytes >= L.total, "head_loss_forward: workspace too small (%lld < %lld)", (long long)workspace_bytes, L.total);
  B200SEG_CHECK_ARG(scratch_bytes >= aspp_yt_bytes(N, C, h, w, R), "head_loss_forward: scratch too small");
  StepKey key = {};
  int np = 0, ni = 0;
  key.p[np++] = x; key.p[np++] = labels; key.p[np++] = workspace; key.p[np++] = scratch; key.p[np++] = logits; key.p[np++] = loss_out;
  B200SEG_CHECK_ARG(R <= 8, "head_loss_forward: %d dilation branches unsupported", R);
  for (int r = 0; r < R; ++r) { key.p[np++] = weights[r]; key.p[np++] = biases ? biases[r] : nullptr; key.i[ni++] = rates_host[r]; }
  const long long ints[] = {1, x_kind, R, N, Cin, C, h, w, label_bytes, H, W, ignore_index, need_grad, workspace_bytes, scratch_bytes};
  for (long long v : ints) key.i[ni++] = v;
  int dev = 0;
  cudaGetDevice(&dev);
  key.i[ni++] = dev;
  key.f[0] = inv_temperature;
  return run_step(key, S(stream), true, [&](cudaStream_t st) -> int {
    char* base = reinterpret_cast<char*>(workspace);
    float* bias_sum = reinterpret_cast<float*>(base + L.bias_sum);
    int rc = aspp_pack_weights(weights, biases, R, C, Cin, base + L.Wp, base + L.WpT, bias_sum, st);
    if (rc) return rc;
    const void* Xp = x;
    if (x_kind == 0) {
      rc = aspp_pack_features(reinterpret_cast<const float*>(x), N, Cin, h, w, base + L.Xp, st);
      if (rc) return rc;
      Xp = base + L.Xp;
    }
    rc = aspp_forward(Xp, base + L.Wp, bias_sum, rates_host, R, N, Cin, C, h, w, reinterpret_cast<float*>(scratch), logits, st);
    if (rc) return rc;
    return k2_forward(logits, N, C, h, w, labels, label_bytes, H, W, ignore_index, inv_temperature, need_grad, base + L.k2ws,
                      k2_workspace_bytes(N, C, h, w, H, W), reinterpret_cast<float*>(base + L.out2), st, loss_out);
  });
}

int b200seg_head_loss_backward(void* workspace, int64_t workspace_bytes, const void* x_bf16, int x_kind, const int* rates_host, int R,
                               int N, int Cin, int C, int h, int w, int H, int W, float inv_temperature, const float* grad_loss,
                               void* scratch, int64_t scratch_bytes, float* grad_x, void* grad_x_nhwc_bf16, float* const* grad_w,
                               float* const* grad_b, void* weights_ready_event, void* stream) {
  REQUIRE_DEVICE();
  B200SEG_CHECK_ARG(workspace && rates_host && scratch, "head_loss_backward: null pointer");
  B200SEG_CHECK_ARG(x_kind == 0 || (x_kind == 1 && (x_bf16 || !grad_w)), "head_loss_backward: bad x_kind / missing bf16 features");
  B200SEG_CHECK_ARG(N > 0 && Cin > 0 && C > 0 && h > 0 && w > 0 && R > 0 && R <= 8 && H > 0 && W > 0, "head_loss_backward: bad shape");
  const HeadLossLayout L = head_loss_layout(N, Cin, C, h, w, R, H, W, x_kind);
  B200SEG_CHECK_ARG(workspace_bytes >= L.total, "head_loss_backward: workspace too small");
  const int splits = head_default_splits((long long)N * h * w, C, Cin, R);
  B200SEG_CHECK_ARG(scratch_bytes >= aspp_bwd_scratch_bytes(N, Cin, C, h, w, R, splits), "head_loss_backward: scratch too small");
  StepKey key = {};
  int np = 0, ni = 0;
  key.p[np++] = workspace; key.p[np++] = x_bf16; key.p[np++] = grad_loss; key.p[np++] = scratch; key.p[np++] = grad_x;
  key.p[np++] = grad_x_nhwc_bf16;
  for (int r = 0; r < R; ++r) { key.p[np++] = grad_w ? grad_w[r] : nullptr; key.p[np++] = grad_b ? grad_b[r] : nullptr; key.i[ni++] = rates_host[r]; }
  const long long ints[] = {2, x_kind, R, N, Cin, C, h, w, H, W, grad_w != nullptr, grad_b != nullptr, workspace_bytes, scratch_bytes};
  for (long long v : ints) key.i[ni++] = v;
  int dev = 0;
  cudaGetDevice(&dev);
  key.i[ni++] = dev;
  key.f[0] = inv_temperature;
  key.p[np++] = weights_ready_event;       // recorded as an external event node inside the graph (aspp_backward_packed)
  return run_step(key, S(stream), true, [&](cudaStream_t st) -> int {
    char* base = reinterpret_cast<char*>(workspace);
    void* gOt = aspp_bwd_gOt_ptr(scratch);
    int rc = k2_backward_packed_multi(base + L.k2ws, N, C, h, w, H, W, inv_temperature, reinterpret_cast<const float*>(base + L.out2),
                                      grad_loss, gOt, grad_b, grad_b ? R : 0, st);
    if (rc) return rc;
    if (!grad_x && !grad_x_nhwc_bf16 && !grad_w) return B200SEG_OK;
    const void* Xp = x_kind == 0 ? static_cast<const void*>(base + L.Xp) : x_bf16;
    return aspp_backward_packed(gOt, Xp, base + L.WpT, rates_host, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, grad_x, grad_w,
                                st, grad_x_nhwc_bf16, reinterpret_cast<cudaEvent_t>(weights_ready_event));
  });
}

// ---------------------------------------------------------------------------------------------------------------------------
// PixelDiscriminator conv stack (discriminator.py:34-47) as ONE call per direction, with the same argument-keyed graph replay as
// the head entries above: weight pack, feature pack and the three conv layers forward; the whole backward chain (gradient layout
// conversion, bias sums, three weight-gradient and three data-gradient GEMMs with their reductions) in the other direction.
// Every buffer is caller-provided (the Python side allocates exactly what the separate entries allocate), so the composition adds
// no arithmetic and no layout of its own: results are bit-identical to the separate entries.
// ---------------------------------------------------------------------------------------------------------------------------
static int round8i(int v) { return (v + 7) / 8 * 8; }

int64_t b200seg_disc_backward_scratch_bytes(int N, int Cin, int h, int w, int ndf1, int ndf2, int C) {
  if (N <= 0 || Cin <= 0 || h <= 0 || w <= 0 || ndf1 <= 0 || ndf2 <= 0 || C <= 0) return 0;
  long long m = nhwc_colsum_scratch_bytes(round8i(2 * C));
  const long long cands[] = {conv3x3_wgrad_scratch_bytes(N, h, w, 2 * C, ndf2, 0), conv3x3_wgrad_scratch_bytes(N, h, w, ndf2, ndf1, 0),
                             conv3x3_wgrad_scratch_bytes(N, h, w, ndf1, Cin, 0), conv3x3_dgrad_colsum_scratch_bytes(N, h, w, ndf2),
                             conv3x3_dgrad_colsum_scratch_bytes(N, h, w, ndf1)};
  for (long long v : cands) m = v > m ? v : m;
  return m + 256;
}

int b200seg_disc_forward(const void* x, int x_kind, int N, int Cin, int h, int w, int ndf1, int ndf2, int C, const float* w1,
                         const float* b1, const float* w2, const float* b2, const float* wc1, const float* bc1, const float* wc2,
                         const float* bc2, float slope, int do_pack, void* Wf1, void* Wb1, void* Wf2, void* Wb2, void* Wf3, void* Wb3,
                         float* b3, void* Xp, void* A1, void* A2, float* out, void* stream) {
  REQUIRE_DEVICE();
  B200SEG_CHECK_ARG(x && Wf1 && Wb1 && Wf2 && Wb2 && Wf3 && Wb3 && b3 && A1 && A2 && out, "disc_forward: null pointer");
  B200SEG_CHECK_ARG(x_kind == 0 || x_kind == 1, "disc_forward: x_kind must be 0 (fp32 NCHW) or 1 (bf16 NHWC), got %d", x_kind);
  B200SEG_CHECK_ARG(x_kind == 1 || Xp, "disc_forward: fp32 NCHW features need the Xp buffer");
  B200SEG_CHECK_ARG(!do_pack || (w1 && w2 && wc1 && wc2), "disc_forward: null weight pointer");
  B200SEG_CHECK_ARG(N > 0 && Cin > 0 && h > 0 && w > 0 && ndf1 > 0 && ndf2 > 0 && C > 0 && Cin % 8 == 0 && ndf1 % 8 == 0 && ndf2 % 8 == 0,
                    "disc_forward: bad shape (channel counts must be multiples of 8)");
  StepKey key = {};
  int np = 0, ni = 0;
  const void* ptrs[] = {x, w1, b1, w2, b2, wc1, bc1, wc2, bc2, Wf1, Wb1, Wf2, Wb2, Wf3, Wb3, b3, Xp, A1, A2, out};
  for (const void* q : ptrs) key.p[np++] = q;
  int dev = 0;
  cudaGetDevice(&dev);
  const long long ints[] = {3, x_kind, N, Cin, h, w, ndf1, ndf2, C, do_pack, dev};
  for (long long v : ints) key.i[ni++] = v;
  key.f[0] = slope;
  return run_step(key, S(stream), true, [&](cudaStream_t st) -> int {
    int rc;
    if (do_pack) {
      const float* weights[4] = {w1, w2, wc1, wc2};
      const int part_co[4] = {ndf1, ndf2, C, C}, parts_per_layer[3] = {1, 1, 2}, cis[3] = {Cin, ndf1, ndf2};
      void* Wfs[3] = {Wf1, Wf2, Wf3};
      void* Wbs[3] = {Wb1, Wb2, Wb3};
      const int pitches[3] = {round8i(ndf1), round8i(ndf2), round8i(2 * C)};
      const float* bias_parts[2] = {bc1, bc2};
      const int bias_lens[2] = {C, C};
      rc = conv3x3_pack_weights_stack(3, weights, part_co, parts_per_layer, cis, Wfs, Wbs, pitches, bias_parts, bias_lens, 2, b3, st);
      if (rc) return rc;
    }
    const void* act = x;
    if (x_kind == 0) {
      rc = aspp_pack_features(reinterpret_cast<const float*>(x), N, Cin, h, w, Xp, st);
      if (rc) return rc;
      act = Xp;
    }
    rc = conv3x3_forward(act, N, h, w, Cin, Cin, Wf1, ndf1, 1, b1, 1, slope, A1, ndf1, nullptr, st);
    if (rc) return rc;
    rc = conv3x3_forward(A1, N, h, w, ndf1, ndf1, Wf2, ndf2, 1, b2, 1, slope, A2, ndf2, nullptr, st);
    if (rc) return rc;
    return conv3x3_forward(A2, N, h, w, ndf2, ndf2, Wf3, 2 * C, 1, b3, 0, 0.f, nullptr, 2 * C, out, st);
  });
}

int b200seg_disc_backward(const float* grad_out, const void* Xp, const void* A1, const void* A2, const void* Wb1, const void* Wb2,
                          const void* Wb3, int N, int Cin, int h, int w, int ndf1, int ndf2, int C, float slope, void* G3, void* dZ2,
                          void* dZ1, void* scratch, int64_t scratch_bytes, float* gw1, float* gb1, float* gw2, float* gb2, float* gwc1,
                          float* gwc2, float* gb3, float* gx_f32_nchw, void* gx_bf16_nhwc, void* stream) {
  REQUIRE_DEVICE();
  B200SEG_CHECK_ARG(grad_out && Xp && A1 && A2 && Wb1 && Wb2 && Wb3 && G3 && scratch, "disc_backward: null pointer");
  B200SEG_CHECK_ARG(N > 0 && Cin > 0 && h > 0 && w > 0 && ndf1 > 0 && ndf2 > 0 && C > 0, "disc_backward: bad shape");
  B200SEG_CHECK_ARG(!(gx_f32_nchw && gx_bf16_nhwc), "disc_backward: give at most one feature-gradient destination");
  const bool need_x = gx_f32_nchw || gx_bf16_nhwc;
  const bool need_l1 = need_x || gw1 || gb1;                 // anything below layer 2's data gradient
  const bool need_l2 = need_l1 || gw2 || gb2;                // anything below layer 3's data gradient
  B200SEG_CHECK_ARG(!need_l2 || dZ2, "disc_backward: dZ2 buffer missing");
  B200SEG_CHECK_ARG(!need_l1 || dZ1, "disc_backward: dZ1 buffer missing");
  B200SEG_CHECK_ARG(scratch_bytes >= b200seg_disc_backward_scratch_bytes(N, Cin, h, w, ndf1, ndf2, C), "disc_backward: scratch too small");
  StepKey key = {};
  int np = 0, ni = 0;
  const void* ptrs[] = {grad_out, Xp, A1, A2, Wb1, Wb2, Wb3, G3, dZ2, dZ1, scratch, gw1, gb1, gw2, gb2, gwc1, gwc2, gb3, gx_f32_nchw, gx_bf16_nhwc};
  for (const void* q : ptrs) key.p[np++] = q;
  int dev = 0;
  cudaGetDevice(&dev);
  const long long ints[] = {4, N, Cin, h, w, ndf1, ndf2, C, scratch_bytes, dev};
  for (long long v : ints) key.i[ni++] = v;
  key.f[0] = slope;
  return run_step(key, S(stream), true, [&](cudaStream_t st) -> int {
    const int p3 = round8i(2 * C);
    int rc = nchw_to_nhwc_bf16(grad_out, N, 2 * C, h * w, G3, p3, st);
    if (rc) return rc;
    if (gb3) {                                                // bias gradient of cls1 | cls2: column sums of the loss gradient
      rc = nhwc_bf16_colsum(G3, (long long)N * h * w, 2 * C, p3, scratch, gb3, st);
      if (rc) return rc;
    }
    if (gwc1 || gwc2) {
      float* outs[2] = {gwc1, gwc2};
      const int parts[2] = {C, C};
      rc = conv3x3_wgrad(G3, 2 * C, p3, A2, ndf2, ndf2, N, h, w, 1, 0, scratch, scratch_bytes, outs, parts, 2, st);
      if (rc) return rc;
    }
    if (!need_l2) return B200SEG_OK;
    // dZ2 = (G3 * Wb3) . LeakyReLU'(A2); the bias gradient of layer 2 comes out of the same epilogue
    rc = conv3x3_dgrad(G3, N, h, w, p3, p3, Wb3, ndf2, 1, A2, slope, dZ2, ndf2, nullptr, st, gb2 ? scratch : nullptr,
                       gb2 ? scratch_bytes : 0, gb2);
    if (rc) return rc;
    if (gw2) {
      float* outs[1] = {gw2};
      const int parts[1] = {ndf2};
      rc = conv3x3_wgrad(dZ2, ndf2, ndf2, A1, ndf1, ndf1, N, h, w, 1, 0, scratch, scratch_bytes, outs, parts, 1, st);
      if (rc) return rc;
    }
    if (!need_l1) return B200SEG_OK;
    rc = conv3x3_dgrad(dZ2, N, h, w, ndf2, ndf2, Wb2, ndf1, 1, A1, slope, dZ1, ndf1, nullptr, st, gb1 ? scratch : nullptr,
                       gb1 ? scratch_bytes : 0, gb1);
    if (rc) return rc;
    if (gw1) {
      float* outs[1] = {gw1};
      const int parts[1] = {ndf1};
      rc = conv3x3_wgrad(dZ1, ndf1, ndf1, Xp, Cin, Cin, N, h, w, 1, 0, scratch, scratch_bytes, outs, parts, 1, st);
      if (rc) return rc;
    }
    if (need_x)
      rc = conv3x3_dgrad(dZ1, N, h, w, ndf1, ndf1, Wb1, Cin, 1, nullptr, slope, gx_bf16_nhwc, Cin, gx_f32_nchw, st, nullptr, 0, nullptr);
    return rc;
  });
}

void b200seg_set_step_graphs(int on) {
  step_graphs_drop();
  g_step_graphs_on = on ? 1 : 0;
  g_step_hits = g_step_captures = 0;
}

void b200seg_step_graph_stats(long long* replays, long long* captures) {
  if (replays) *replays = g_step_hits;
  if (captures) *captures = g_step_captures;
}

}  // extern "C"
