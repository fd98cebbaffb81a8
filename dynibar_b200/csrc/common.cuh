// Shared helpers for the dynibar_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "dynibar_b200.h"

namespace dyn {

// thread-local error string behind dyn_last_error()
char* err_buf();
int fail(int code, const char* fmt, ...);

#define DYN_CHECK_ARG(cond)                                                    \
  do {                                                                         \
    if (!(cond))                                                               \
      return dyn::fail(DYN_E_INVALID, "%s:%d: argument check failed: %s",      \
                       __FILE__, __LINE__, #cond);                             \
  } while (0)

#define DYN_CUDA(call)                                                         \
  do {                                                                         \
    cudaError_t e_ = (call);                                                   \
    if (e_ != cudaSuccess)                                                     \
      return dyn::fail(DYN_E_CUDA, "%s:%d: %s: %s", __FILE__, __LINE__, #call, \
                       cudaGetErrorString(e_));                                \
  } while (0)

// every kernel launch of the library goes through this macro; the counter backs
// dyn_launch_count() (bench.py's `gpu_launches`)
extern unsigned long long g_launches;
#define DYN_LAUNCH_CHECK()            \
  do {                                \
    ++dyn::g_launches;                \
    DYN_CUDA(cudaGetLastError());     \
  } while (0)

// ---- optional per-kernel-class device timing (dyn_profile_*): CUDA events on the
// launching stream around the big fused kernels; off by default.
enum ProfClass { PROF_VIEW_ST = 0, PROF_VIEW_DY, PROF_MOTION, PROF_POINT1, PROF_POINT2, PROF_RGBHEAD,
                 PROF_ATTENTION, PROF_GATHER, PROF_NCLASS };
void prof_begin(int cls, cudaStream_t st);
void prof_end(int cls, cudaStream_t st);
struct ProfScope {
  int cls; cudaStream_t st;
  ProfScope(int c, cudaStream_t s) : cls(c), st(s) { prof_begin(c, s); }
  ~ProfScope() { prof_end(cls, st); }
};

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

constexpr int kC = 32;      // feature channels (coarse_feat_dim / fine_feat_dim)
constexpr int kF = kC + 3;  // gathered channels per view
constexpr int kMaxViews = 32;

// ---- network parameter layout (flat fp32 blob; offsets in floats) ----------
// Order = dynibar_b200/weights.py CANONICAL_ORDER[kind].
struct LinearP {
  int w;  // offset of weight [out, in]
  int b;  // offset of bias [out] or -1
  int in, out;
  long long tc;  // byte offset of the packed tensor-core image in dyn_net::packed
};
struct LayerList {
  LinearP l[32];
  int n;
  long long packed_bytes;
};

struct DynamicLayout {
  LinearP ray_dir0, ray_dir2, base0, base2, vis0, vis2, vis2_0, vis2_2, geo0, geo2;
  LinearP wq, wk, wv, fc;
  int ln_w, ln_b;
  LinearP refpts0, refpts2, outgeo0, outgeo2, rgb0, rgb2, rgb4;
  int total;
  LayerList all;
};
struct StaticLayout {
  int s;  // scalar anti-alias parameter (present iff anti_alias_pooling)
  LinearP ray_dir0, ray_dir2, ref_feat, base0, base2, vis0, vis2, vis2_0, vis2_2, geo0, geo2;
  LinearP wq, wk, wv, fc;
  int ln_w, ln_b;
  LinearP outgeo0, outgeo2, rgb0, rgb2, rgb4;
  int total;
  LayerList all;
};
struct MotionLayout {
  LinearP pts[8];
  LinearP coeff;
  int total;
  LayerList all;
};

DynamicLayout dynamic_layout();
StaticLayout static_layout(bool anti_alias);
MotionLayout motion_layout(int nb);

struct FusedChunk;
struct ChainImage {
  const void* img;
  const FusedChunk* tab;
  int nchunks;
};

}  // namespace dyn

struct dyn_net {
  int kind;
  const float* params;  // caller-owned flat fp32 blob (device)
  void* packed;         // caller-owned tensor-core operand images (device) or null
  int n_samples;
  float shift;
  int anti_alias;
  int mask_rgb;
  int nb;  // motion: number of basis functions
  dyn::DynamicLayout dl;
  dyn::StaticLayout sl;
  dyn::MotionLayout ml;
  // motion net: the whole MotionMLP as one fused chain (chains_fused.cu)
  dyn::ChainImage motion;
  // aggregation nets, twin-warp row-local chains (chains_twin.cu): [0] point stage 1, [1] point stage 2,
  // [2] static blending head
  dyn::ChainImage chain_tw[3];
  // aggregation nets, per-view stage (view_twin3.cu): weight images in its column layout
  dyn::ChainImage twin3;
};

// ---- device helpers ---------------------------------------------------------
__device__ __forceinline__ float elu_f(float x) { return x > 0.f ? x : expm1f(x); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }
// torch Softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// F.normalize(v, dim=-1): v / max(||v||, 1e-12)
__device__ __forceinline__ void normalize3(float& x, float& y, float& z) {
  float n = sqrtf(x * x + y * y + z * z);
  float inv = 1.f / fmaxf(n, 1e-12f);
  x *= inv; y *= inv; z *= inv;
}
