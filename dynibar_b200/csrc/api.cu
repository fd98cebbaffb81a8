// C ABI glue: error reporting, network handles, precision dispatch.
#include <stdarg.h>
#include <stdlib.h>

#include <vector>

#include "linear_tc.cuh"
#include "nets.cuh"
#include "nets_fused.cuh"

namespace dyn {

unsigned long long g_launches = 0;

// ---- profiling hook ----
static int g_prof_on = 0;
struct ProfPair { cudaEvent_t a, b; int cls; };
static std::vector<ProfPair> g_prof;
static cudaEvent_t g_prof_open[PROF_NCLASS];

void prof_begin(int cls, cudaStream_t st) {
  if (!g_prof_on) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  g_prof_open[cls] = e;
}
void prof_end(int cls, cudaStream_t st) {
  if (!g_prof_on || !g_prof_open[cls]) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  g_prof.push_back(ProfPair{g_prof_open[cls], e, cls});
  g_prof_open[cls] = nullptr;
}

char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

}  // namespace dyn

using namespace dyn;

extern "C" {

int dyn_version(void) { return 100; }

unsigned long long dyn_launch_count(int reset) {
  unsigned long long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

const char* dyn_last_error(void) { return err_buf(); }

int dyn_device_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  return n;
}

void dyn_profile_enable(int on) {
  g_prof_on = on;
  if (on) {
    for (auto& p : g_prof) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    g_prof.clear();
  }
}

int dyn_profile_read(int cls, float* total_ms, int* launches) {
  DYN_CHECK_ARG(cls >= 0 && cls < PROF_NCLASS && total_ms && launches);
  float tot = 0.f;
  int n = 0;
  for (auto& p : g_prof) {
    if (p.cls != cls) continue;
    DYN_CUDA(cudaEventSynchronize(p.b));
    float ms = 0.f;
    DYN_CUDA(cudaEventElapsedTime(&ms, p.a, p.b));
    tot += ms;
    ++n;
  }
  *total_ms = tot;
  *launches = n;
  return DYN_OK;
}

size_t dyn_net_param_count(int kind) {
  switch (kind) {
    case DYN_NET_DYNAMIC: return (size_t)dynamic_layout().total;
    case DYN_NET_STATIC: return (size_t)static_layout(true).total;  // with `s`; without = count - 1
    case DYN_NET_MOTION: return (size_t)motion_layout(6).total;
    default: return 0;
  }
}

size_t dyn_net_packed_bytes(int kind) {
  switch (kind) {
    case DYN_NET_DYNAMIC: return (size_t)dynamic_layout().all.packed_bytes + view_twin3_bytes(kind) + twin_chain_bytes(kind);
    case DYN_NET_STATIC: return (size_t)static_layout(true).all.packed_bytes + view_twin3_bytes(kind) + twin_chain_bytes(kind);
    case DYN_NET_MOTION: return (size_t)motion_layout(8).all.packed_bytes + fused_chain_bytes(kind);
    default: return 0;
  }
}

size_t dyn_net_layer_images_bytes(int kind) {
  switch (kind) {
    case DYN_NET_DYNAMIC: return (size_t)dynamic_layout().all.packed_bytes;
    case DYN_NET_STATIC: return (size_t)static_layout(true).all.packed_bytes;
    case DYN_NET_MOTION: return (size_t)motion_layout(8).all.packed_bytes;
    default: return 0;
  }
}

int dyn_net_create(int kind, const float* params, size_t n_params, void* packed, int n_samples,
                   float shift, int anti_alias_pooling, int mask_rgb, void* stream, dyn_net_t* out) {
  return dyn_net_create_ex(kind, params, n_params, packed, packed != nullptr ? 2 : 0, n_samples, shift,
                           anti_alias_pooling, mask_rgb, stream, out);
}

int dyn_net_create_ex(int kind, const float* params, size_t n_params, void* packed, int pack_level, int n_samples,
                      float shift, int anti_alias_pooling, int mask_rgb, void* stream, dyn_net_t* out) {
  DYN_CHECK_ARG(out != nullptr && params != nullptr);
  DYN_CHECK_ARG(pack_level >= 0 && pack_level <= 2 && (pack_level == 0 || packed != nullptr));
  if (pack_level == 0) packed = nullptr;
  dyn_net* n = (dyn_net*)calloc(1, sizeof(dyn_net));
  if (!n) return fail(DYN_E_INVALID, "out of host memory");
  n->kind = kind;
  n->params = params;
  n->packed = packed;
  n->n_samples = n_samples;
  n->shift = shift;
  n->anti_alias = anti_alias_pooling;
  n->mask_rgb = mask_rgb;
  size_t expect = 0;
  if (kind == DYN_NET_DYNAMIC) {
    n->dl = dynamic_layout();
    expect = n->dl.total;
  } else if (kind == DYN_NET_STATIC) {
    n->sl = static_layout(anti_alias_pooling != 0);
    expect = n->sl.total;
  } else if (kind == DYN_NET_MOTION) {
    // coeff_linear is [3*nb, 256] + [3*nb]: solve nb from the count
    size_t fixed = (size_t)motion_layout(1).total - (3 * 256 + 3);
    size_t rest = n_params - fixed;
    if (n_params <= fixed || rest % (3 * 257) != 0) {
      free(n);
      return fail(DYN_E_INVALID, "MotionMLP: unexpected parameter count %zu", n_params);
    }
    n->nb = (int)(rest / (3 * 257));
    if (n->nb < 1 || n->nb > 8) {
      free(n);
      return fail(DYN_E_INVALID, "MotionMLP: num_basis %d unsupported (1..8)", n->nb);
    }
    n->ml = motion_layout(n->nb);
    expect = n->ml.total;
  } else {
    free(n);
    return fail(DYN_E_INVALID, "unknown net kind %d", kind);
  }
  if (expect != n_params) {
    free(n);
    return fail(DYN_E_INVALID, "net kind %d: got %zu parameters, expected %zu", kind, n_params, expect);
  }
  if (packed != nullptr) {  // tensor-core operand images of every layer
    const LayerList& ll = kind == DYN_NET_DYNAMIC ? n->dl.all : (kind == DYN_NET_STATIC ? n->sl.all : n->ml.all);
    for (int i = 0; i < ll.n; ++i) {
      int rc = tc_pack_weight(params + ll.l[i].w, ll.l[i].out, ll.l[i].in,
                              reinterpret_cast<char*>(packed) + ll.l[i].tc, (cudaStream_t)stream);
      if (rc) { free(n); return rc; }
    }
    if (pack_level >= 2) {  // fused tensor-core images (per-view stage, row-local chains): packed on the host once
      float* hp = (float*)malloc(n_params * sizeof(float));
      if (!hp) { free(n); return fail(DYN_E_INVALID, "out of host memory"); }
      cudaError_t e = cudaMemcpyAsync(hp, params, n_params * sizeof(float), cudaMemcpyDeviceToHost,
                                      (cudaStream_t)stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
      int rc = e == cudaSuccess ? DYN_OK : fail(DYN_E_CUDA, "reading parameters back: %s", cudaGetErrorString(e));
      char* cur = reinterpret_cast<char*>(packed) + ll.packed_bytes;
      if (!rc && kind == DYN_NET_MOTION) {
        rc = fused_chain_build(n, hp, cur, fused_chain_bytes(kind), (cudaStream_t)stream);
      } else if (!rc) {
        rc = view_twin3_build(n, hp, cur, view_twin3_bytes(kind), (cudaStream_t)stream);
        cur += view_twin3_bytes(kind);
        if (!rc) rc = twin_chain_build(n, hp, cur, twin_chain_bytes(kind), (cudaStream_t)stream);
      }
      free(hp);
      if (rc) { free(n); return rc; }
    }
  }
  *out = n;
  return DYN_OK;
}

void dyn_net_destroy(dyn_net_t net) { free(net); }

size_t dyn_motion_workspace_bytes(int R, int S) { return motion_f32_workspace((long long)R * S); }

size_t dyn_net_workspace_bytes(int kind, int R, int S, int V) {
  if (kind == DYN_NET_DYNAMIC) return net_dynamic_f32_workspace(R, S, V);
  if (kind == DYN_NET_STATIC) return net_static_f32_workspace(R, S, V);
  if (kind == DYN_NET_MOTION) return motion_f32_workspace((long long)R * S);
  return 0;
}

size_t dyn_net_fused_workspace_bytes(int kind, int R, int S, int V) {
  return net_fused_workspace(kind, R, S, V);
}

int dyn_featmaps_channels_last(const float* featmaps, void* out_bf16, int V, int C, int h, int w,
                               void* stream) {
  DYN_CHECK_ARG(featmaps && out_bf16 && V >= 1 && C >= 1 && h >= 1 && w >= 1);
  return launch_to_channels_last_bf16(featmaps, out_bf16, V, C, h * w, (cudaStream_t)stream);
}

int dyn_rgbs_rgba(const float* src_rgbs, float* out_rgba, int V, int H, int W, void* stream) {
  DYN_CHECK_ARG(src_rgbs && out_rgba && V >= 1 && H >= 1 && W >= 1);
  return launch_rgb_to_rgba(src_rgbs, out_rgba, (long long)V * H * W, (cudaStream_t)stream);
}

void dyn_debug_set_view_kernel(int which) { set_view_kernel(which); }

static long long* g_view_dbg = nullptr;
void dyn_debug_set_view_timestamps(long long* dev_buf) { g_view_dbg = dev_buf; }
long long* view_dbg_ptr() { return g_view_dbg; }

int dyn_net_static_fused(dyn_net_t net, const float* pts, const float* ray_o, const float* ray_d,
                         const float* query_cam, const float* src_rgbs, const float* src_cams,
                         const void* feat_cl, int R, int S, int V, int H, int W, int C, int h, int w,
                         float* raw, float* mask_out, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (R == 0) return DYN_OK;  // empty batch: nothing to do (pointers may be null)
  DYN_CHECK_ARG(net && net->kind == DYN_NET_STATIC && pts && ray_o && ray_d && query_cam && src_rgbs);
  DYN_CHECK_ARG(src_cams && feat_cl && raw && mask_out && workspace && C == kC);
  DYN_CHECK_ARG(R >= 0 && S >= 1 && V >= 1 && V <= 16);
  if (R == 0) return DYN_OK;
  return net_static_fused(net, pts, ray_o, ray_d, query_cam, src_rgbs, src_cams, feat_cl, R, S, V, H, W,
                          h, w, raw, mask_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int dyn_net_dynamic_fused(dyn_net_t net, const float* pts, const float* pts_seq, const float* ray_dir,
                          const float* query_cam, const float* src_rgbs, const float* src_cams,
                          const void* feat_cl, float time, int R, int S, int V, int H, int W, int C,
                          int h, int w, float* raw, float* mask_out, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (R == 0) return DYN_OK;  // empty batch: nothing to do (pointers may be null)
  DYN_CHECK_ARG(net && net->kind == DYN_NET_DYNAMIC && pts && pts_seq && ray_dir && query_cam);
  DYN_CHECK_ARG(src_rgbs && src_cams && feat_cl && raw && mask_out && workspace && C == kC);
  DYN_CHECK_ARG(R >= 0 && S >= 1 && V >= 1 && V <= 16);
  if (R == 0) return DYN_OK;
  return net_dynamic_fused(net, pts, pts_seq, ray_dir, query_cam, src_rgbs, src_cams, feat_cl, time, R, S,
                           V, H, W, h, w, raw, mask_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int dyn_debug_point_chain(dyn_net_t net, const float* G, const float* nvalid, const float* pts,
                          const float* ray_dir, int R, int S, float* g2, float* Q, float* K, float* V,
                          float* O, float* out_a, float* out_b, float* posenc_ws, void* stream) {
  DYN_CHECK_ARG(net && G && nvalid && g2 && Q && K && V && O && out_a && posenc_ws);
  return debug_point_chain(net, G, nvalid, pts, ray_dir, R, S, g2, Q, K, V, O, out_a, out_b, posenc_ws,
                           (cudaStream_t)stream);
}

int dyn_debug_pack_layer(const float* W, const float* bias, int N, int Kw, int Npad, int Kpad,
                         const int* colmap, float scale, int stage_bytes, void* out_img, size_t out_bytes,
                         size_t* img_bytes, int* nchunks) {
  DYN_CHECK_ARG(W && colmap && out_img && img_bytes && nchunks);
  return debug_pack_layer(W, bias, N, Kw, Npad, Kpad, colmap, scale, stage_bytes, out_img, out_bytes, img_bytes,
                          nchunks);
}
size_t dyn_debug_tile_image_off(long long row, int kgroup, int kgroups) {
  return debug_tile_image_off(row, kgroup, kgroups);
}

int dyn_motion_coeffs(dyn_net_t motion, const float* pts, float time, int R, int S, float* coeff,
                      void* workspace, size_t workspace_bytes, int precision, void* stream) {
  if (R == 0) return DYN_OK;  // empty batch: nothing to do (pointers may be null)
  DYN_CHECK_ARG(motion && motion->kind == DYN_NET_MOTION && pts && coeff && workspace);
  DYN_CHECK_ARG(R >= 0 && S >= 1);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = motion_f32(motion, pts, 3, false, time, (long long)R * S, coeff, workspace, workspace_bytes, precision, st);
  if (rc) return rc;
  return zero_last_samples(coeff, R, S, 3 * motion->nb, st);
}

int dyn_motion_mlp(dyn_net_t motion, const float* xyzt, int N, float* coeff, void* workspace,
                   size_t workspace_bytes, int precision, void* stream) {
  DYN_CHECK_ARG(motion && motion->kind == DYN_NET_MOTION && xyzt && coeff && workspace && N >= 0);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  return motion_f32(motion, xyzt, 4, true, 0.f, N, coeff, workspace, workspace_bytes, precision,
                    (cudaStream_t)stream);
}

size_t dyn_motion_train_workspace_bytes(int N) { return motion_train_workspace(N < 0 ? 0 : N); }

int dyn_motion_mlp_train_forward(dyn_net_t motion, const float* xyzt, int N, float* coeff, void* saved,
                                 size_t saved_bytes, int precision, void* stream) {
  DYN_CHECK_ARG(motion && motion->kind == DYN_NET_MOTION && N >= 0);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  if (N == 0) return DYN_OK;
  DYN_CHECK_ARG(xyzt && coeff && saved);
  return motion_train_forward(motion, xyzt, N, coeff, saved, saved_bytes, precision, (cudaStream_t)stream);
}

int dyn_motion_mlp_backward(dyn_net_t motion, const float* xyzt, const float* d_coeff, int N, void* saved,
                            size_t saved_bytes, float* d_params, float* d_xyzt, int precision, void* stream) {
  DYN_CHECK_ARG(motion && motion->kind == DYN_NET_MOTION && N >= 0);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  if (N == 0) return DYN_OK;
  DYN_CHECK_ARG(xyzt && d_coeff && saved && d_params);
  return motion_train_backward(motion, xyzt, d_coeff, N, saved, saved_bytes, d_params, d_xyzt, precision,
                               (cudaStream_t)stream);
}

int dyn_net_dynamic(dyn_net_t net, const float* pts, const float* rgb_feat, const float* ray_dir,
                    const float* mask, float time, int R, int S, int V, float* raw, void* workspace,
                    size_t workspace_bytes, int precision, void* stream) {
  if (R == 0) return DYN_OK;  // empty batch: nothing to do (pointers may be null)
  DYN_CHECK_ARG(net && net->kind == DYN_NET_DYNAMIC && pts && rgb_feat && ray_dir && mask && raw);
  DYN_CHECK_ARG(workspace && R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  return net_dynamic_f32(net, pts, rgb_feat, ray_dir, mask, time, R, S, V, raw, workspace,
                         workspace_bytes, precision, (cudaStream_t)stream);
}

int dyn_net_static(dyn_net_t net, const float* pts, const float* ref_rays, const float* src_rays,
                   const float* rgb_feat, const float* ray_diff, const float* mask, int R, int S, int V,
                   float* raw, void* workspace, size_t workspace_bytes, int precision, void* stream) {
  if (R == 0) return DYN_OK;  // empty batch: nothing to do (pointers may be null)
  DYN_CHECK_ARG(net && net->kind == DYN_NET_STATIC && pts && ref_rays && src_rays && rgb_feat);
  DYN_CHECK_ARG(ray_diff && mask && raw && workspace && R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  return net_static_f32(net, pts, ref_rays, src_rays, rgb_feat, ray_diff, mask, R, S, V, raw, workspace,
                        workspace_bytes, precision, (cudaStream_t)stream);
}

size_t dyn_net_train_workspace_bytes(int kind, int R, int S, int V) {
  if (kind != DYN_NET_DYNAMIC && kind != DYN_NET_STATIC) return 0;
  return net_train_workspace(kind, R, S, V);
}

size_t dyn_net_backward_scratch_bytes(int kind, int R, int S, int V) {
  if (kind != DYN_NET_DYNAMIC && kind != DYN_NET_STATIC) return 0;
  return net_backward_scratch(kind, R, S, V);
}

int dyn_net_dynamic_train_forward(dyn_net_t net, const float* pts, const float* rgb_feat, const float* ray_dir,
                                  const float* mask, float time, int R, int S, int V, float* raw, void* saved,
                                  size_t saved_bytes, int precision, void* stream) {
  if (R == 0) return DYN_OK;
  DYN_CHECK_ARG(net && net->kind == DYN_NET_DYNAMIC && pts && rgb_feat && ray_dir && mask && raw && saved);
  DYN_CHECK_ARG(R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  if (precision == DYN_PREC_BF16 && net->packed == nullptr)
    return fail(DYN_E_INVALID, "bf16 training needs a net created with layer images (dyn_net_create_ex, pack_level >= 1)");
  return net_dynamic_f32(net, pts, rgb_feat, ray_dir, mask, time, R, S, V, raw, saved, saved_bytes, precision,
                         (cudaStream_t)stream, /*train=*/true);
}

int dyn_net_dynamic_backward(dyn_net_t net, const float* pts, const float* mask, int R, int S, int V,
                             const float* d_raw, void* saved, size_t saved_bytes, void* scratch,
                             size_t scratch_bytes, float* d_params, float* d_rgb_feat, float* d_pts, int precision,
                             void* stream) {
  if (R == 0) return DYN_OK;
  DYN_CHECK_ARG(net && net->kind == DYN_NET_DYNAMIC && pts && mask && d_raw && saved && scratch && d_params);
  DYN_CHECK_ARG(R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  return net_dynamic_backward(net, pts, nullptr, nullptr, mask, R, S, V, d_raw, saved, saved_bytes, scratch,
                              scratch_bytes, d_params, d_rgb_feat, d_pts, precision, (cudaStream_t)stream);
}

int dyn_net_static_train_forward(dyn_net_t net, const float* pts, const float* ref_rays, const float* src_rays,
                                 const float* rgb_feat, const float* ray_diff, const float* mask, int R, int S,
                                 int V, float* raw, void* saved, size_t saved_bytes, int precision, void* stream) {
  if (R == 0) return DYN_OK;
  DYN_CHECK_ARG(net && net->kind == DYN_NET_STATIC && pts && ref_rays && src_rays && rgb_feat);
  DYN_CHECK_ARG(ray_diff && mask && raw && saved && R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  if (precision == DYN_PREC_BF16 && net->packed == nullptr)
    return fail(DYN_E_INVALID, "bf16 training needs a net created with layer images (dyn_net_create_ex, pack_level >= 1)");
  return net_static_f32(net, pts, ref_rays, src_rays, rgb_feat, ray_diff, mask, R, S, V, raw, saved, saved_bytes,
                        precision, (cudaStream_t)stream, /*train=*/true);
}

int dyn_net_static_backward(dyn_net_t net, const float* rgb_feat, const float* ray_diff, int R, int S, int V,
                            const float* d_raw, void* saved, size_t saved_bytes, void* scratch,
                            size_t scratch_bytes, float* d_params, float* d_rgb_feat, int precision, void* stream) {
  if (R == 0) return DYN_OK;
  DYN_CHECK_ARG(net && net->kind == DYN_NET_STATIC && rgb_feat && ray_diff && d_raw && saved && scratch && d_params);
  DYN_CHECK_ARG(R >= 0 && S >= 1 && V >= 1 && V <= kMaxViews);
  DYN_CHECK_ARG(precision == DYN_PREC_FP32 || precision == DYN_PREC_BF16);
  return net_static_backward(net, rgb_feat, ray_diff, R, S, V, d_raw, saved, saved_bytes, scratch, scratch_bytes,
                             d_params, d_rgb_feat, precision, (cudaStream_t)stream);
}

}  // extern "C"
