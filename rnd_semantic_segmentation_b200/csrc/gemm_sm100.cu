// Host side of the tcgen05 GEMM core: TMA tensor-map encoding, launch, and an on-device self-test
// against a naive CUDA-core kernel (used by tests/ to pin descriptors on real hardware).
#include <stdlib.h>
#include "gemm_sm100.cuh"
#include <limits.h>

namespace b200seg {
namespace gemm {

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 tensor map: inner (contiguous) extent `inner`, outer extent `outer`, outer pitch in elements.
static int make_tmap(CUtensorMap* m, const __nv_bfloat16* ptr, long long inner, long long outer, long long pitch,
                     int box_inner, int box_outer) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available (driver too old or no GPU)");
    return B200SEG_ERR_CUDA;
  }
  B200SEG_CHECK_ARG((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand pointer must be 16-byte aligned");
  B200SEG_CHECK_ARG((pitch * 2) % 16 == 0, "TMA operand pitch (%lld elements) must be a multiple of 8", pitch);
  cuuint64_t gdim[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t gstride[1] = {(cuuint64_t)pitch * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner=%lld outer=%lld pitch=%lld box=%dx%d)", (int)r,
              inner, outer, pitch, box_inner, box_outer);
    return B200SEG_ERR_CUDA;
  }
  return B200SEG_OK;
}

static int g_overlap_sms = 8;         // b200seg_gemm_set_overlap_sms(): SMs left free while an all-reduce overlaps the dgrad GEMM
void set_overlap_sms(int n) { g_overlap_sms = n < 0 ? 0 : n; }
int overlap_sms() { return g_overlap_sms; }
// b200seg_gemm_set_sharing(): 0 one CTA per tile; 1 (default) what each caller asks for -- cta_group::2 pairs for the forward,
// weight-gradient and seam-format data-gradient GEMMs, 2-CTA multicast pairs for the fp32 NCHW data gradient; 2 = 1 (it named
// 2 x 2 clusters, which measured ~1.9x slower: 37 four-CTA clusters do not all fit the GPCs); 3 = 1 with the fp32 data gradient
// as cta_group::2 pairs too (measured 5 us slower: it is store-bound); 4 = every shared GEMM as cta_group::2 pairs; 5 = no
// cta_group::2 (each caller's pair_fallback: the multicast pairs of the earlier rounds)
static int g_share_enabled = 1;
void set_sharing(int on) { g_share_enabled = on; }

static int g_dgrad_mode = 1;         // b200seg_gemm_set_dgrad_mode(): see gemm_sm100.cuh
void set_dgrad_mode(int mode) { g_dgrad_mode = mode; }
int dgrad_mode() { return g_dgrad_mode; }
static int g_fwd_mode = 1;           // b200seg_gemm_set_fwd_mode(): see gemm_sm100.cuh
void set_fwd_mode(int mode) { g_fwd_mode = mode; }
int fwd_mode() { return g_fwd_mode; }
static int g_narrow_tiles = 1;        // b200seg_gemm_set_narrow_tiles(): 0 = always 256-column tiles
void set_narrow_tiles(int on) { g_narrow_tiles = on; }

// the register-store epilogue that also writes each 32-pixel lane group's per-column (mean, M2) (Out::F32_NCHW_ROWS_STATS)
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_stats_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                       const __grid_constant__ CUtensorMap tmap_out, const Params p) {
  gemm_bf16_body<false, false, SHARE_PAIR, 256, true, false, true>(tmap_a, tmap_b, tmap_out, p);
}

// Every instantiation of gemm_bf16_kernel that launch() can run
typedef void (*KernelFn)(CUtensorMap, CUtensorMap, CUtensorMap, Params);
struct Variant {
  bool a_mn, b_mn;
  int share, bn;
  bool rs, seam, stats;
  KernelFn fn;
  bool configured;
};
template <bool A_MN, bool B_MN, int SHARE, int BN = 256, bool RS = false, bool SEAM = false>
static Variant variant() { return {A_MN, B_MN, SHARE, BN, RS, SEAM, false, gemm_bf16_kernel<A_MN, B_MN, SHARE, BN, RS, SEAM>, false}; }
static Variant g_variants[] = {
    // any operand layout, any sharing geometry, 256-column tiles
    variant<false, false, SHARE_NONE>(), variant<false, false, SHARE_B>(), variant<false, false, SHARE_A>(), variant<false, false, SHARE_PAIR>(),
    variant<true, true, SHARE_NONE>(), variant<true, true, SHARE_B>(), variant<true, true, SHARE_A>(), variant<true, true, SHARE_PAIR>(),
    variant<true, false, SHARE_NONE>(), variant<true, false, SHARE_B>(), variant<true, false, SHARE_A>(), variant<true, false, SHARE_PAIR>(),
    variant<false, true, SHARE_NONE>(), variant<false, true, SHARE_B>(), variant<false, true, SHARE_A>(), variant<false, true, SHARE_PAIR>(),
    // narrow tiles: K-major operands, unshared B
    variant<false, false, SHARE_NONE, 224>(), variant<false, false, SHARE_NONE, 192>(),
    variant<false, false, SHARE_A, 224>(), variant<false, false, SHARE_A, 192>(),
    // fp32 NCHW rows-as-pixels stored from registers, seven ring stages: cta_group::2 pairs, B K-major
    variant<false, false, SHARE_PAIR, 256, true>(), variant<true, false, SHARE_PAIR, 256, true>(),
    // seam epilogue: K-major operands
    variant<false, false, SHARE_NONE, 256, false, true>(), variant<false, false, SHARE_PAIR, 256, false, true>(),
    // fp32 NCHW rows-as-pixels with per-lane-group column statistics: cta_group::2 pairs, K-major operands
    {false, false, SHARE_PAIR, 256, true, false, true, gemm_bf16_stats_kernel, false},
};

static int check(const Gemm& g) {
  const Out& o = g.out;
  const bool aligned = (reinterpret_cast<uintptr_t>(o.ptr) & 15) == 0;
  if (o.layout == Out::SEAM) {
    B200SEG_CHECK_ARG(g.M > 0 && g.N > 0 && g.K > 0 && o.hw > 0 && (g.M % o.hw == 0 || g.M <= o.hw) && g.splits <= 1,
                      "gemm seam: bad problem %dx%dx%d (hw %d)", g.M, g.N, g.K, o.hw);
    B200SEG_CHECK_ARG(!g.a.mn_major && !g.b.mn_major, "gemm seam: K-major operands only");
    B200SEG_CHECK_ARG(o.identity && o.scale && o.bias && g.N % 8 == 0 && aligned,
                      "gemm seam: N = %d must be a multiple of 8 and D 16-byte aligned", g.N);
    return B200SEG_OK;
  }
  if (o.layout == Out::F32_NCHW_ROWS_STATS) {
    B200SEG_CHECK_ARG(g.M > 0 && g.N > 0 && g.K > 0 && o.hw > 0 && (g.M % o.hw == 0 || g.M <= o.hw) && g.splits <= 1,
                      "gemm rows + stats: bad problem %dx%dx%d (hw %d)", g.M, g.N, g.K, o.hw);
    B200SEG_CHECK_ARG(!g.a.mn_major && !g.b.mn_major, "gemm rows + stats: K-major operands only");
    B200SEG_CHECK_ARG(o.stats && (reinterpret_cast<uintptr_t>(o.stats) & 7) == 0, "gemm rows + stats: stats must be 8-byte aligned");
    return B200SEG_OK;
  }
  B200SEG_CHECK_ARG(g.M > 0 && g.N > 0 && g.K > 0, "gemm: empty problem %dx%dx%d", g.M, g.N, g.K);
  B200SEG_CHECK_ARG(o.layout != Out::F32_NCHW_COLS || o.hw > 0, "gemm: the NCHW column map needs hw > 0");
  B200SEG_CHECK_ARG(o.layout != Out::F32_NCHW_ROWS || (o.hw > 0 && g.splits <= 1 && (g.M % o.hw == 0 || g.M <= o.hw)),
                    "gemm: the pixel-major epilogue needs fp32 output, no split-K and whole images (or one plane) along M");
  B200SEG_CHECK_ARG(o.layout != Out::BF16 || (g.N % 8 == 0 && o.row_stride % 8 == 0 && o.split_stride % 8 == 0 && aligned),
                    "gemm: bf16 output needs plain row-major D with N, row pitch multiples of 8 and a 16-byte aligned base");
  return B200SEG_OK;
}

int launch(const Gemm& g, cudaStream_t stream) {
  if (int rc = check(g)) return rc;
  const Operand &a = g.a, &b = g.b;
  const Out& o = g.out;
  const int M = g.M, N = g.N, K = g.K;
  const bool seam = o.layout == Out::SEAM, stats = o.layout == Out::F32_NCHW_ROWS_STATS;
  // callers name the sharing geometry they want; the global mode (A/B experiments) can veto or override it
  int share = g.share;
  if (!g_share_enabled) share = SHARE_NONE;
  if (g_share_enabled == 3 && share == SHARE_B) share = SHARE_PAIR;         // also the store-bound fp32 dgrad as 2-SM pairs
  if (g_share_enabled == 4 && (share == SHARE_A || share == SHARE_B)) share = SHARE_PAIR;
  if (g_share_enabled == 5 && share == SHARE_PAIR) share = g.pair_fallback;
  if (stats) share = SHARE_PAIR;          // its only kernel, under every sharing mode and for a single M-tile too
  Params p = {};
  p.M = M; p.N = N; p.K = K;
  p.m_tiles = ceil_div(M, BLOCK_M);
  p.n_tiles = ceil_div(N, BLOCK_N);
  p.kb_total = ceil_div(K, BLOCK_K);
  const int splits = g.splits < 1 ? 1 : (g.splits > p.kb_total ? p.kb_total : g.splits);
  p.kb_per_split = ceil_div(p.kb_total, splits);
  p.splits = ceil_div(p.kb_total, p.kb_per_split);     // every split non-empty
  if (g.splits_used) *g.splits_used = p.splits;
  p.out = reinterpret_cast<float*>(o.ptr);
  p.row_stride = o.row_stride;
  p.col_hw = o.layout == Out::F32_NCHW_COLS ? o.hw : INT_MAX;
  p.img_stride = o.img_stride;
  p.split_stride = o.split_stride;
  p.out_bf16 = o.layout == Out::BF16 || seam ? 1 : 0;
  // tile order: the units running together should share the LARGER operand, so that it streams from HBM once and the small
  // one lives in L2.  Channel-major problems (M = channels / packed weight rows <= N = pixels) walk along M; pixel-major ones
  // (M = pixels: the seam-format and the register-store data gradients) walk along N -- M-fastest made them re-read the
  // 86 MB pixel operand once per N-tile (653 MB of DRAM reads per launch at the bench shape, ncu profiles/r2_dgrad_*).
  p.n_fastest = M > N ? 1 : 0;
  p.vec_ok = (reinterpret_cast<uintptr_t>(o.ptr) & 15) == 0 && o.row_stride % 4 == 0 && o.split_stride % 4 == 0 &&
             (p.col_hw == INT_MAX || (p.col_hw % 4 == 0 && o.img_stride % 4 == 0));
  if (o.layout == Out::F32_NCHW_ROWS) {
    // every rows-as-pixels launch (the head's pixel-major forward and data gradient, conv3's data gradient) takes
    // b200seg_gemm_set_dgrad_mode(2)'s streaming stores and the B200SEG_EPI_SLEEP pacing (<ns> after each 16-column chunk's stores,
    // default off): with a six-stage ring, spreading a tile's 128 KB of stores over the tile time took the data gradient from 161
    // to 150 us (the store bursts delay the operand requests queued behind them); with the seventh stage it no longer changes
    // anything (154-156 us with 0 or 192 ns), so it stays an experiment knob
    static int env_ns = -2;
    if (env_ns == -2) { const char* e = getenv("B200SEG_EPI_SLEEP"); env_ns = e ? atoi(e) : 0; }
    p.row_hw_px = o.hw;
    p.row_hw = g_dgrad_mode == 2 ? 2 : 1;
    p.epi_sleep_ns = env_ns > 0 ? env_ns : 0;
  } else if (stats) {
    // conv3 under batch statistics: the register-store epilogue with plain stores, no pacing
    p.row_hw_px = o.hw;
    p.row_hw = 1;
    p.stats = o.stats;
  } else if (seam) {
    // the fused conv3 + tail of the backbone's last Bottleneck: pairs along M walking along N, so a pair's two pixel tiles are read
    // once for all N-tiles while the small weight operand stays in L2
    p.row_stride = N;
    p.img_stride = (long long)N * o.hw;
    p.row_hw_px = o.hw;
    p.n_fastest = 1;
    p.vec_ok = 0;
    p.seam_identity = o.identity;
    p.seam_scale = o.scale;
    p.seam_bias = o.bias;
  }
  // a pair needs two tiles along the paired dimension to be worth it
  if (share == SHARE_B && p.m_tiles < 2) share = SHARE_NONE;
  if (share == SHARE_PAIR && p.m_tiles < 2 && !stats) share = SHARE_NONE;
  if (share == SHARE_A && p.n_tiles < 2) share = SHARE_NONE;

  // tile width: with K-major operands, fp32 output and an unshared B tile, a narrower tile that makes the tile count a
  // near-multiple of the worker count beats 256 columns (rounds x columns is the cost)
  int bn = BLOCK_N;
  if (g_narrow_tiles && !a.mn_major && !b.mn_major && !p.out_bf16 && (share == SHARE_NONE || share == SHARE_A)) {
    const int workers = share == SHARE_A ? num_sms() / 2 : num_sms();
    long long best = -1;
    for (int cand : {256, 224, 192}) {
      const int nt = ceil_div(N, cand);
      if (share == SHARE_A && nt < 2) continue;
      const long long units = (long long)p.m_tiles * (share == SHARE_A ? (nt + 1) / 2 : nt) * p.splits;
      const long long cost = ceil_div_ll(units, workers) * cand;
      if (best < 0 || cost < best) { best = cost; bn = cand; }
    }
    p.n_tiles = ceil_div(N, bn);
  }
  const bool rs = p.row_hw == 1 && share == SHARE_PAIR && !b.mn_major;        // register-store variant (7 ring stages)
  Variant* v = nullptr;
  for (Variant& c : g_variants)
    if (c.a_mn == a.mn_major && c.b_mn == b.mn_major && c.share == share && c.bn == bn && c.rs == rs && c.seam == seam &&
        c.stats == stats) { v = &c; break; }
  B200SEG_CHECK_ARG(v, "gemm: no kernel for operands %d/%d, sharing %d, %d-column tiles, output layout %d", (int)a.mn_major,
                    (int)b.mn_major, share, bn, (int)o.layout);

  // the shared operand is loaded in halves (one per CTA of the pair): halve its K-major box
  CUtensorMap ta, tb;
  int rc;
  if (!a.mn_major) rc = make_tmap(&ta, a.ptr, K, M, a.pitch, BLOCK_K, share == SHARE_A ? BLOCK_M / 2 : BLOCK_M);
  else rc = make_tmap(&ta, a.ptr, M, K, a.pitch, 64, BLOCK_K);
  if (rc) return rc;
  if (!b.mn_major) rc = make_tmap(&tb, b.ptr, K, N, b.pitch, BLOCK_K, (share == SHARE_B || share == SHARE_PAIR) ? BLOCK_N / 2 : bn);
  else rc = make_tmap(&tb, b.ptr, N, K, b.pitch, 64, BLOCK_K);
  if (rc) return rc;
  CUtensorMap to = ta;            // third tensor-map slot: the 64-row B boxes of the register-store variant (below)
  if (rs) {
    rc = make_tmap(&to, b.ptr, K, N, b.pitch, BLOCK_K, BLOCK_N / 4);          // 64-row B boxes for a ragged last N-tile
    if (rc) return rc;
  }

  // persistent CTAs, one per SM, minus the SMs the caller wants left free for a concurrent kernel (the NCCL all-reduce
  // of the weight gradients running underneath the data-gradient GEMM)
  int sms = num_sms() - (g.sm_reserve > 0 ? g.sm_reserve : 0);
  if (sms < 2) sms = 2;
  const int cs = share == SHARE_NONE ? 1 : 2;                                 // CTAs per cluster
  const int mt = (share == SHARE_B || share == SHARE_PAIR) ? (p.m_tiles + 1) / 2 : p.m_tiles;
  const int nt = share == SHARE_A ? (p.n_tiles + 1) / 2 : p.n_tiles;
  const int units = mt * nt * p.splits;
  const int grid = cs * (units < sms / cs ? units : sms / cs);

  if (!v->configured) {
    B200SEG_CUDA(cudaFuncSetAttribute(v->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    v->configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = share == SHARE_NONE ? 0 : 1;
  profile_begin(g.prof_tag, stream);
  B200SEG_CUDA(cudaLaunchKernelEx(&cfg, v->fn, ta, tb, to, p));
  B200SEG_LAUNCH_CHECK();
  profile_end(g.prof_tag, stream);
  return B200SEG_OK;
}

// ------------------------------------------------------------------------------------------
// forward GEMM with the fp32 NCHW -> bf16 conversion of the pixel operand inside the kernel
// ------------------------------------------------------------------------------------------
// b200seg_gemm_set_fwd_convert(): 1 = the head's forward takes fp32 NCHW features through gemm_fwd_convert_kernel where eligible.
// Default 0: measured EQUAL to pack + plain GEMM at the eval shape (158.8 vs 158.3 us per 1 x 2048 x 128 x 256 frame) -- a ring
// stage is converted only after it has been released, so convert + proxy fence + cluster-scope publish (~2.5 us, most of it the
// fence waiting for the remote stores) sits in every stage's critical path; see DESIGN.md for what would remove it.
static int g_fwd_convert = 0;
void set_fwd_convert(int on) { g_fwd_convert = on; }

bool fwd_convert_eligible(const float* x, int K, int hw, int M) {
  const int m_pairs = (ceil_div(M, BLOCK_M) + 1) / 2;
  return g_fwd_convert && g_share_enabled != 0 && x != nullptr && hw > 0 && hw % 4 == 0 && K % BLOCK_K == 0 && M > BLOCK_M &&
         m_pairs <= FWDX_MAX_MP && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
}

template <int MP>
static int launch_fwd_convert_t(const CUtensorMap& ta, const FwdXParams& p, cudaStream_t stream, int prof_tag) {
  static bool configured = false;
  static int max_clusters = 0;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(FWDX_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2 * MP;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (!configured) {
    B200SEG_CUDA(cudaFuncSetAttribute(gemm_fwd_convert_kernel<MP>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    // how many clusters of this size the device can hold at once (GPC granularity): the grid is sized to it
    cfg.gridDim = dim3(2 * MP * (num_sms() / (2 * MP)));
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, gemm_fwd_convert_kernel<MP>, &cfg) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = num_sms() / (2 * MP);
    }
    max_clusters = n;
    configured = true;
  }
  const int clusters = p.n_tiles < max_clusters ? p.n_tiles : max_clusters;
  cfg.gridDim = dim3(2 * MP * clusters);
  profile_begin(prof_tag, stream);
  B200SEG_CUDA(cudaLaunchKernelEx(&cfg, gemm_fwd_convert_kernel<MP>, ta, p));
  profile_end(prof_tag, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int launch_fwd_convert(const __nv_bfloat16* a, long long a_pitch, const float* x, int n_img, int hw, int M, int K, float* out,
                       long long row_stride, __nv_bfloat16* xn, cudaStream_t stream, int prof_tag) {
  B200SEG_CHECK_ARG(fwd_convert_eligible(x, K, hw, M), "gemm: forward-with-conversion called on an ineligible shape");
  B200SEG_CHECK_ARG(xn == nullptr || (reinterpret_cast<uintptr_t>(xn) & 15) == 0, "gemm: the bf16 feature copy must be 16-byte aligned");
  const long long P = (long long)n_img * hw;
  B200SEG_CHECK_ARG(P < (1LL << 31), "gemm: too many pixels");
  FwdXParams p;
  p.M = M; p.P = (int)P; p.K = K;
  p.m_tiles = ceil_div(M, BLOCK_M);
  p.n_tiles = ceil_div((int)P, BLOCK_N);
  p.kb_total = K / BLOCK_K;
  p.out = out; p.row_stride = row_stride;
  p.x = x; p.hw = hw; p.xn = xn;
  CUtensorMap ta;
  int rc = make_tmap(&ta, a, K, M, a_pitch, BLOCK_K, BLOCK_M);
  if (rc) return rc;
  switch ((p.m_tiles + 1) / 2) {
    case 1: return launch_fwd_convert_t<1>(ta, p, stream, prof_tag);
    case 2: return launch_fwd_convert_t<2>(ta, p, stream, prof_tag);
    default: return launch_fwd_convert_t<3>(ta, p, stream, prof_tag);
  }
}

// ------------------------------------------------------------------------------------------
// Self-test helpers
// ------------------------------------------------------------------------------------------
__global__ void fill_bf16_kernel(__nv_bfloat16* p, long long n, uint32_t seed) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x = (uint32_t)i * 2654435761u + seed;
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  p[i] = __float2bfloat16(((float)(x & 0xFFFF) / 65536.0f - 0.5f) * 2.0f);
}

__global__ void naive_gemm_kernel(const __nv_bfloat16* A, const __nv_bfloat16* B, float* C, int M, int N, int K, int a_mn,
                                  int b_mn, long long a_pitch, long long b_pitch) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  int m = blockIdx.y;
  if (n >= N || m >= M) return;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) {
    float a = __bfloat162float(a_mn ? A[(long long)k * a_pitch + m] : A[(long long)m * a_pitch + k]);
    float b = __bfloat162float(b_mn ? B[(long long)k * b_pitch + n] : B[(long long)n * b_pitch + k]);
    acc = fmaf(a, b, acc);
  }
  C[(long long)m * N + n] = acc;
}

// max |D - ref| and max |ref| over the (possibly split / image-mapped) output
__global__ void compare_kernel(const float* D, const float* ref, int M, int N, int splits, long long split_stride,
                               long long row_stride, int col_hw, long long img_stride, float* out2) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  int m = blockIdx.y;
  if (n >= N || m >= M) return;
  int img = n / col_hw;
  long long off = (long long)img * img_stride + (long long)m * row_stride + (n - img * col_hw);
  float v = 0.f;
  for (int z = 0; z < splits; ++z) v += D[z * split_stride + off];
  float r = ref[(long long)m * N + n];
  atomicMax(reinterpret_cast<int*>(out2), __float_as_int(fabsf(v - r)));
  atomicMax(reinterpret_cast<int*>(out2) + 1, __float_as_int(fabsf(r)));
}

int selftest(int M, int N, int K, int a_mn, int b_mn, int splits, int col_hw, int share, double* max_err, double* max_ref) {
  const long long a_pitch = a_mn ? ((M + 7) / 8) * 8 : ((K + 7) / 8) * 8;
  const long long b_pitch = b_mn ? ((N + 7) / 8) * 8 : ((K + 7) / 8) * 8;
  const long long a_elems = a_pitch * (a_mn ? K : M), b_elems = b_pitch * (b_mn ? K : N);
  __nv_bfloat16 *A = nullptr, *B = nullptr;
  float *D = nullptr, *ref = nullptr, *res = nullptr;
  const int kb_total = ceil_div(K, BLOCK_K);
  int s = splits < 1 ? 1 : (splits > kb_total ? kb_total : splits);
  long long row_stride, img_stride = 0, out_elems;
  if (col_hw > 0) {                       // "NCHW" map: column n -> image n / col_hw, D[img][row][col % hw]
    const int imgs = ceil_div(N, col_hw);
    row_stride = col_hw;
    img_stride = (long long)M * col_hw;
    out_elems = (long long)imgs * img_stride;
  } else {
    row_stride = ((N + 3) / 4) * 4;
    out_elems = (long long)M * row_stride;
  }
  B200SEG_CUDA(cudaMalloc(&A, a_elems * 2));
  B200SEG_CUDA(cudaMalloc(&B, b_elems * 2));
  B200SEG_CUDA(cudaMalloc(&D, out_elems * 4 * s));
  B200SEG_CUDA(cudaMalloc(&ref, (long long)M * N * 4));
  B200SEG_CUDA(cudaMalloc(&res, 8));
  B200SEG_CUDA(cudaMemset(res, 0, 8));
  B200SEG_CUDA(cudaMemset(D, 0xFF, out_elems * 4 * s));      // NaN pattern: unwritten outputs are caught
  fill_bf16_kernel<<<(unsigned)ceil_div_ll(a_elems, 256), 256>>>(A, a_elems, 1234u);
  fill_bf16_kernel<<<(unsigned)ceil_div_ll(b_elems, 256), 256>>>(B, b_elems, 777u);
  dim3 g(ceil_div(N, 128), M);
  naive_gemm_kernel<<<g, 128>>>(A, B, ref, M, N, K, a_mn, b_mn, a_pitch, b_pitch);
  B200SEG_LAUNCH_CHECK();
  Operand oa{A, a_mn != 0, a_pitch}, ob{B, b_mn != 0, b_pitch};
  int used = 1;
  Gemm gm{oa, ob, M, N, K,
          col_hw > 0 ? out_f32_nchw_cols(D, col_hw, row_stride, img_stride, out_elems) : out_f32(D, row_stride, out_elems)};
  gm.splits = s;
  gm.splits_used = &used;
  gm.share = share == 3 ? SHARE_A : share;      // 3 named the 2 x 2-cluster geometry, which was removed: it runs as SHARE_A
  int rc = launch(gm, 0);
  if (rc == B200SEG_OK) {
    compare_kernel<<<g, 128>>>(D, ref, M, N, used, out_elems, row_stride, col_hw > 0 ? col_hw : INT_MAX, img_stride, res);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      set_error("gemm selftest: kernel failed: %s", cudaGetErrorString(e));
      rc = B200SEG_ERR_CUDA;
    } else {
      float h[2];
      cudaMemcpy(h, res, 8, cudaMemcpyDeviceToHost);
      // a NaN difference compares as a huge positive int pattern -> report as inf
      *max_err = (h[0] != h[0]) ? 1e30 : (double)h[0];
      *max_ref = (double)h[1];
    }
  }
  cudaFree(A); cudaFree(B); cudaFree(D); cudaFree(ref); cudaFree(res);
  return rc;
}

// ---- self-test of the forward-with-conversion kernel: fp32 NCHW x, reference on bf16-rounded x; also checks the bf16 copy ----
__global__ void fill_f32_kernel(float* p, long long n, uint32_t seed) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x = (uint32_t)i * 2654435761u + seed;
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  p[i] = ((float)(x & 0xFFFFFF) / 16777216.0f - 0.5f) * 2.0f;
}
__global__ void naive_fwdx_kernel(const __nv_bfloat16* A, const float* x, float* C, int M, int P, int K, int hw, long long a_pitch) {
  int pcol = blockIdx.x * blockDim.x + threadIdx.x;
  int m = blockIdx.y;
  if (pcol >= P || m >= M) return;
  const int img = pcol / hw, off = pcol - img * hw;
  float acc = 0.f;
  for (int k = 0; k < K; ++k)
    acc = fmaf(__bfloat162float(A[(long long)m * a_pitch + k]), __bfloat162float(__float2bfloat16(x[((long long)img * K + k) * hw + off])), acc);
  C[(long long)m * P + pcol] = acc;
}
__global__ void compare_xn_kernel(const float* x, const __nv_bfloat16* xn, long long n, float* out1) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float d = fabsf(__bfloat162float(xn[i]) - __bfloat162float(__float2bfloat16(x[i])));
  if (!(d == 0.f)) atomicMax(reinterpret_cast<int*>(out1), __float_as_int(d != d ? 1e30f : d));
}

int selftest_fwd_convert(int M, int n_img, int hw, int K, int write_xn, double* max_err, double* max_ref, double* xn_err) {
  const long long P = (long long)n_img * hw;
  const long long a_pitch = K, xe = (long long)n_img * K * hw;
  const long long row_stride = ((P + 3) / 4) * 4;
  __nv_bfloat16 *A = nullptr, *xn = nullptr;
  float *x = nullptr, *D = nullptr, *ref = nullptr, *res = nullptr;
  B200SEG_CUDA(cudaMalloc(&A, (long long)M * a_pitch * 2));
  B200SEG_CUDA(cudaMalloc(&x, xe * 4));
  B200SEG_CUDA(cudaMalloc(&xn, xe * 2));
  B200SEG_CUDA(cudaMalloc(&D, (long long)M * row_stride * 4));
  B200SEG_CUDA(cudaMalloc(&ref, (long long)M * P * 4));
  B200SEG_CUDA(cudaMalloc(&res, 16));
  B200SEG_CUDA(cudaMemset(res, 0, 16));
  B200SEG_CUDA(cudaMemset(D, 0xFF, (long long)M * row_stride * 4));
  B200SEG_CUDA(cudaMemset(xn, 0xFF, xe * 2));
  fill_bf16_kernel<<<(unsigned)ceil_div_ll((long long)M * a_pitch, 256), 256>>>(A, (long long)M * a_pitch, 4321u);
  fill_f32_kernel<<<(unsigned)ceil_div_ll(xe, 256), 256>>>(x, xe, 99u);
  dim3 g(ceil_div((int)P, 128), M);
  naive_fwdx_kernel<<<g, 128>>>(A, x, ref, M, (int)P, K, hw, a_pitch);
  B200SEG_LAUNCH_CHECK();
  int rc = launch_fwd_convert(A, a_pitch, x, n_img, hw, M, K, D, row_stride, write_xn ? xn : nullptr, 0, -1);
  if (rc == B200SEG_OK) {
    compare_kernel<<<g, 128>>>(D, ref, M, (int)P, 1, 0, row_stride, INT_MAX, 0, res);
    if (write_xn) compare_xn_kernel<<<(unsigned)ceil_div_ll(xe, 256), 256>>>(x, xn, xe, res + 2);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      set_error("gemm fwd-convert selftest: kernel failed: %s", cudaGetErrorString(e));
      rc = B200SEG_ERR_CUDA;
    } else {
      float h[3];
      cudaMemcpy(h, res, 12, cudaMemcpyDeviceToHost);
      *max_err = (h[0] != h[0]) ? 1e30 : (double)h[0];
      *max_ref = (double)h[1];
      *xn_err = (double)h[2];
    }
  }
  cudaFree(A); cudaFree(x); cudaFree(xn); cudaFree(D); cudaFree(ref); cudaFree(res);
  return rc;
}

}  // namespace gemm
}  // namespace b200seg
