// Tile geometry and workspace layout shared by the K2 kernels (ce_kernels.cu: the generic CTA-tile kernel;
// ce_v2_kernels.cu: the warp-tile kernel for the common upsampling ratios) and their finalize kernels.
#pragma once
#include "common.cuh"

namespace b200seg {

struct K2Geom {
  int N, C, h, w, H, W;
  int tile_w, tile_h;           // output pixels per tile (128 x 32 CTA tiles, or 32 x 32 warp tiles)
  int tiles_x, tiles_y;
  int ispan_max, jspan_max;     // max number of source rows / cols touched by one tile
  int kmax;                     // max number of tile columns that interpolate from one source column
  float scale_h, scale_w;
};

__host__ __device__ __forceinline__ int host_i0(float scale, int dst) { return (int)(scale * (float)dst); }

inline void k2_geometry_tiled(K2Geom& g, int N, int C, int h, int w, int H, int W, int tile_w, int tile_h) {
  g.N = N; g.C = C; g.h = h; g.w = w; g.H = H; g.W = W;
  g.tile_w = tile_w; g.tile_h = tile_h;
  g.tiles_x = ceil_div(W, tile_w);
  g.tiles_y = ceil_div(H, tile_h);
  g.scale_h = ac_scale(h, H);
  g.scale_w = ac_scale(w, W);
  g.ispan_max = 1; g.jspan_max = 1;
  for (int ty = 0; ty < g.tiles_y; ++ty) {
    const int ya = ty * tile_h, yb = (ya + tile_h < H ? ya + tile_h : H) - 1;
    const int lo = host_i0(g.scale_h, ya);
    int hi = host_i0(g.scale_h, yb); hi += (hi < h - 1) ? 1 : 0;
    if (hi - lo + 1 > g.ispan_max) g.ispan_max = hi - lo + 1;
  }
  for (int tx = 0; tx < g.tiles_x; ++tx) {
    const int xa = tx * tile_w, xb = (xa + tile_w < W ? xa + tile_w : W) - 1;
    const int lo = host_i0(g.scale_w, xa);
    int hi = host_i0(g.scale_w, xb); hi += (hi < w - 1) ? 1 : 0;
    if (hi - lo + 1 > g.jspan_max) g.jspan_max = hi - lo + 1;
  }
  // longest run of output columns sharing one x0, doubled (+2): columns with x0 in {j-1, j} feed source column j
  int run = 0, best = 1, prev = -1;
  for (int x = 0; x < W; ++x) {
    const int i0 = host_i0(g.scale_w, x);
    run = (i0 == prev) ? run + 1 : 1;
    prev = i0;
    if (run > best) best = run;
  }
  g.kmax = 2 * best + 2;
  if (g.kmax > tile_w) g.kmax = tile_w;
}

// Workspace layout (floats): [tiles] loss partial | [tiles] valid-count partial | [tiles][ispan][jspan][C] blocks |
// bias partials | 256 spare bytes (the warp-tile kernel keeps its dynamic tile counter in the first 4 of them)
inline long long k2_block_floats(const K2Geom& g) { return (long long)g.ispan_max * g.jspan_max * g.C; }
inline long long k2_tiles(const K2Geom& g) { return (long long)g.N * g.tiles_x * g.tiles_y; }
// per finalize-block partial sums of the low-res gradient (bias gradient), [N*h*ceil(w/128)][32]
inline long long k2_bias_part_floats(const K2Geom& g) { return (long long)g.N * g.h * ceil_div(g.w, 128) * 32; }
inline long long k2_geom_bytes(const K2Geom& g) {
  return (2 * k2_tiles(g) + k2_tiles(g) * k2_block_floats(g) + k2_bias_part_floats(g)) * 4 + 256;
}

struct K2Params {
  K2Geom g;
  const float* logits;       // [N,C,h,w]
  const void* labels;        // [N,H,W] int64, or uint8 when label_u8
  int label_u8;
  int ignore_index;
  float inv_T;
  float* loss_part;          // [tiles]
  float* cnt_part;           // [tiles]
  float* blocks;             // [tiles][ispan_max][jspan_max][C]
  unsigned* counter;         // warp-tile kernel: dynamic tile counter (zeroed by the launcher)
};

// ce_v2_kernels.cu
constexpr int K2V2_SPAN = 8;          // source columns a 32-column warp tile may touch
bool k2v2_eligible(int N, int C, int h, int w, int H, int W);
void k2v2_geometry(K2Geom& g, int N, int C, int h, int w, int H, int W);
int k2v2_main_launch(const K2Params& p, bool grad, cudaStream_t stream);

}  // namespace b200seg
