// Fused per-view tensor-core stage (nets_fused.cu): argument block + host API.
#pragma once
#include <cuda_bf16.h>

#include "geometry.cuh"

namespace dyn {

constexpr int kGStride = 272;  // row stride of the pooled per-point feature G (257 used)

struct FusedChunk {
  uint32_t off, bytes;   // weight chunk inside the image
  uint16_t npad;         // UMMA N of the layer
  uint8_t ksteps;        // K = 16 * ksteps in this chunk
  uint8_t flags;         // 1: wait for the operand (a_ready) before this chunk
                         // 2: last chunk of a round (signal the epilogue)
                         // 8: first k-step overwrites D (start of a layer)
  uint16_t a_kgroup;     // first 8-column group of the A tile this chunk consumes
  uint16_t d_col;        // accumulator column offset inside the tile's TMEM region
};

struct ViewFusedArgs {
  // inputs
  const float* pts;       // [P,3] reference-time sample points
  const float* pts_seq;   // motion-displaced points, view v at pts_seq + v*seq_stride*3 (dynamic) or null
  long long seq_stride;
  const float* rgba;      // [V,H,W,4] fp32 source images, alpha = 0 (dyn_rgbs_rgba)
  const uint16_t* feat_bf;  // [V,h,w,32] channels-last bf16 feature maps (dyn_featmaps_channels_last)
  const float* ref_feat;  // [R,35] static: ref_feature_fc(PE(ref plucker)) per ray
  const float* dfeat;     // [35] dynamic: time feature
  const float* params;    // fp32 parameter blob (biases, small heads)
  const void* wimg;       // packed weight chunks
  const FusedChunk* chunks;
  int nchunks;
  ViewCams cams;
  float h_img, w_img;
  int H, W, h, w, V, S;
  long long P;
  int anti_alias, mask_rgb;
  int o_b1, o_b2, o_b3, o_b4, o_b5, o_b6, o_w6, o_b7, o_w8, o_b8, o_s;
  // outputs
  float* G;          // [P, kGStride]: mean128 | var128 | mean weight
  float* nvalid;     // [P]
  float* mask_proj;  // [P*V] projector mask (in front & in bounds)
  float* mask_eff;   // static [P*V]: mask after mask_rgb gating
  float* X;          // static [P*V,128] **bf16** (declared float* for the workspace): per-view feature after the visibility residual
  float* vis2;       // static [P*V]
  float* ray_diff;   // static [P*V,4]
  float* rgb_in;     // static [P*V,3] gathered source colours
  int producers;     // lanes of the producer warp that stream weight chunks (1 or 2)
  int ablate;        // profiling only (DYN_ABLATE): 1 skip gather loads, 2 skip X/vis/mask stores, 4 skip pooled-output stores, 8 skip second pooling
  long long* dbg;    // optional: clock64() phase timestamps of block 0 (profiling builds/tests only)
};

// ---- row-local fused chains: MotionMLP (chains_fused.cu), point stages and blending head (chains_twin.cu) ----
struct MotionFusedArgs {
  const float* x;  // [N, ldx] xyz (+ time column when time_is_column)
  int ldx, time_is_column;
  float time;
  long long N;
  int S, n_last;   // zero the last n_last samples of each S-sample ray (S = 0: never)
  float* coeff;    // [N, ncoef]
  int ncoef;
  const float* params;
  int o_bias[9];
  const void* wimg;
  const FusedChunk* chunks;
  int nchunks;
  int producers;  // lanes of the producer warp that stream weight chunks
};

struct Point1Args {
  const float* G;       // [P, kGStride]
  const float* posenc;  // [S,128] sinusoid table (dynamic) or null
  long long P;
  int S;
  float* g2;                 // [P,128] fp32 (residual of the ray transformer)
  __nv_bfloat16 *Q, *K, *V;  // [P,128] bf16 (operands of the attention)
  const float* params;
  int o_bgeo0, o_bgeo2;
  const void* wimg;
  const FusedChunk* chunks;
  int nchunks;
  int producers;  // lanes of the producer warp that stream weight chunks
};

struct Point2Args {
  const __nv_bfloat16* O;  // [P,128] bf16 attention output
  const float* g2;      // [P,128] residual
  const float* nvalid;  // [P]
  const float* pts;     // [P,3]   (dynamic)
  const float* ray_dir; // [R,3]   (dynamic)
  long long P;
  int S;
  float shift;
  float* raw;    // dynamic: [P,4]
  float* GW;     // static:  [P,128] per-point part of rgb_fc.0 (bias included)
  float* sigma;  // static:  [P] masked density
  const float* params;
  int o_lnw, o_lnb, o_brefpts0, o_brefpts2, o_boutgeo0, o_woutgeo2, o_boutgeo2, o_brgb0, o_brgb2,
      o_wrgb4, o_brgb4;
  const void* wimg;
  const FusedChunk* chunks;
  int nchunks;
  int producers;  // lanes of the producer warp that stream weight chunks
};

struct RgbHeadArgs {
  const float *X /* bf16 tile image, 16 k-groups, rows = view slots (point * VP + view) */, *vis2, *ray_diff, *mask_eff, *rgb_in, *GW, *sigma;
  long long P;
  int V;
  float* raw;  // [P,4]
  const float* params;
  int o_brgb2, o_wrgb4, o_brgb4;
  const void* wimg;
  const FusedChunk* chunks;
  int nchunks;
  int producers;  // lanes of the producer warp that stream weight chunks
};

int debug_pack_layer(const float* W, const float* bias, int N, int Kw, int Npad, int Kpad, const int* colmap,
                     float scale, int stage_bytes, void* out_img, size_t out_bytes, size_t* img_bytes,
                     int* nchunks);
size_t debug_tile_image_off(long long row, int kgroup, int kgroups);
size_t fused_chain_bytes(int kind);
int fused_chain_build(dyn_net* n, const float* host_params, void* dst_dev, size_t dst_bytes,
                      cudaStream_t st);
int launch_motion_fused(const dyn_net* n, MotionFusedArgs& a, cudaStream_t st);

// twin-warp row-local chains (chains_twin.cu)
size_t twin_chain_bytes(int kind);
int twin_chain_build(dyn_net* n, const float* host_params, void* dst_dev, size_t dst_bytes, cudaStream_t st);
int launch_point1_twin(const dyn_net* n, Point1Args& a, cudaStream_t st);
int launch_point2_twin(const dyn_net* n, Point2Args& a, cudaStream_t st);
int launch_rgbhead_twin(const dyn_net* n, RgbHeadArgs& a, cudaStream_t st);

// sub-round pipelined twin-warp per-view stage (view_twin3.cu)
size_t view_twin3_bytes(int kind);
int view_twin3_build(dyn_net* n, const float* host_params, void* dst_dev, size_t dst_bytes, cudaStream_t st);
int launch_view_twin3(const dyn_net* n, ViewFusedArgs& a, int V, cudaStream_t st);

void set_view_kernel(int which);
int producer_lanes();  // DYN_PRODUCERS (default 1)
int launch_view_fused(const dyn_net* n, ViewFusedArgs& a, int V, cudaStream_t st);

}  // namespace dyn
