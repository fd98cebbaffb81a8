/* dynibar_b200 -- C ABI of the B200-native DynIBaR per-ray IBR hot path.
 *
 * The reference (google/dynibar @ 5412b55) has no FFI layer: its boundary for
 * this path is the Python call surface of ibrnet/render_ray.py,
 * ibrnet/projection.py and ibrnet/mlp_network.py.  Each entry point below
 * names the reference function (file:line under /root/reference) it replaces;
 * the Python modules under dynibar_b200/ bind them with ctypes behind the reference's own
 * function / class names (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *     tensors are dense row-major fp32 unless stated; shapes in comments.
 *     The tiny per-frame arrays (`*_cam`, `*_cams`, `basis`) may be HOST
 *     pointers as well: host copies are read without synchronising the stream.
 *   - the caller owns every buffer (inputs, outputs, workspace, packed
 *     weights); the library never allocates or frees device memory and keeps
 *     no device pointer after return except inside a `dyn_net_t` handle.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it,
 *     nothing synchronises.
 *   - return 0 on success, a negative DYN_E_* otherwise; `dyn_last_error()`
 *     returns a thread-local message.  No C++ exceptions cross the ABI.
 *   - R rays, S samples per ray, V source views, C feature channels (32),
 *     F = C + 3.
 */
#ifndef DYNIBAR_B200_H_
#define DYNIBAR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DYN_OK 0
#define DYN_E_INVALID -1 /* bad argument / unsupported shape */
#define DYN_E_CUDA -2    /* a CUDA runtime call or launch failed */
#define DYN_E_WORKSPACE -3 /* workspace too small */

#define DYN_NET_DYNAMIC 0 /* DynibarDynamic, mlp_network.py:129 */
#define DYN_NET_STATIC 1  /* DynibarStatic,  mlp_network.py:319 */
#define DYN_NET_MOTION 2  /* MotionMLP,      mlp_network.py:558 */

#define DYN_PREC_FP32 0 /* SIMT fp32 everywhere (parity mode) */
#define DYN_PREC_BF16 1 /* tcgen05: bf16 operands, fp32 accumulate/statistics */

typedef struct dyn_net* dyn_net_t;

int dyn_version(void);
const char* dyn_last_error(void);
/* Number of SMs etc. of the current device (for grid sizing diagnostics). */
int dyn_device_sm_count(void);
/* Kernels launched by this library since load (or the last reset). */
unsigned long long dyn_launch_count(int reset);

/* (debug / measurement hooks below -- dyn_profile_*, dyn_debug_*, dyn_launch_count -- keep process-global
 * state and are NOT thread-safe; the entry points of the path itself only touch caller-owned buffers.) */
/* Optional device timing of the big kernels (CUDA events on the launching
 * stream, recorded inside the library around each launch).  Classes: 0 fused
 * static per-view stage, 1 fused dynamic per-view stage, 2 MotionMLP, 3 point
 * stage 1, 4 point stage 2, 5 static blending head, 6 ray-transformer attention,
 * 7 stand-alone projection+gather.  enable(1) clears previous records. */
void dyn_profile_enable(int on);
int dyn_profile_read(int cls, float* total_ms, int* launches);

/* ---- weights ------------------------------------------------------------
 * `params` is the flat fp32 concatenation of the network's state_dict tensors
 * in the canonical order documented in dynibar_b200/weights.py (reference key
 * names, mlp_network.py:159-214 / :349-403 / :591-603).  `n_params` is checked
 * against the expected count.  `packed` is a caller-owned device buffer of
 * dyn_net_packed_bytes(kind) bytes that receives the tensor-core operand
 * images (bf16, UMMA canonical layout); it may be NULL for DYN_PREC_FP32 use.
 * n_samples sizes the sinusoid table of the dynamic net (mlp_network.py:218).
 */
size_t dyn_net_param_count(int kind);
size_t dyn_net_packed_bytes(int kind);
int dyn_net_create(int kind, const float* params, size_t n_params, void* packed,
                   int n_samples, float shift, int anti_alias_pooling,
                   int mask_rgb, void* stream, dyn_net_t* out);
/* pack_level: 0 = fp32 parameters only (packed may be NULL), 1 = per-layer tensor-core images only
 * (dyn_net_layer_images_bytes(kind) bytes: enough for the staged DYN_PREC_BF16 evaluation and the bf16 training
 * step, cheap enough to rebuild after every optimizer step), 2 = everything (== dyn_net_create). */
size_t dyn_net_layer_images_bytes(int kind);
int dyn_net_create_ex(int kind, const float* params, size_t n_params, void* packed, int pack_level,
                      int n_samples, float shift, int anti_alias_pooling, int mask_rgb, void* stream,
                      dyn_net_t* out);
void dyn_net_destroy(dyn_net_t net);

/* ---- a2: sample_along_camera_ray, render_ray.py:67-131 -------------------
 * ray_o, ray_d [R,3]; jitter [R,S] of U[0,1) or NULL (det=True).
 * Outputs pts [R,S,3], z_vals [R,S], s_vals [R,S]. */
int dyn_sample_rays(const float* ray_o, const float* ray_d, float near_depth,
                    float far_depth, int R, int S, int inv_uniform,
                    const float* jitter, float* pts, float* z_vals,
                    float* s_vals, void* stream);

/* pts = z * d + o and s = z_to_s(z) for given depths
 * (render_ray.py:822-831, :399-404).  s_vals may be NULL. */
int dyn_points_from_depths(const float* ray_o, const float* ray_d,
                           const float* z_vals, float near_depth,
                           float far_depth, int R, int S, float* pts,
                           float* s_vals, void* stream);

/* ---- a3: MotionMLP + trajectory displacement ------------------------------
 * mlp_network.py:605-618; render_ray.py:361-369, :462-500.
 * coeff [R,S,3*nb] with the last round(0.1*S) samples zeroed. */
size_t dyn_motion_workspace_bytes(int R, int S);
int dyn_motion_coeffs(dyn_net_t motion, const float* pts, float time, int R,
                      int S, float* coeff, void* workspace,
                      size_t workspace_bytes, int precision, void* stream);
/* generic MotionMLP forward on xyzt rows [N,4] -> [N,3*nb]
 * (MotionMLP.forward, no zeroing). */
int dyn_motion_mlp(dyn_net_t motion, const float* xyzt, int N, float* coeff,
                   void* workspace, size_t workspace_bytes, int precision,
                   void* stream);
/* pts_seq[v] = pts + traj(frame+off_v) - traj(frame) for the n_off temporal
 * offsets, followed by num_vv copies of pts.  basis [T,nb] (model.py:18-30).
 * offsets_host is a HOST array.  pts_seq [n_off+num_vv, R, S, 3]. */
int dyn_traj_displace(const float* pts, const float* coeff, const float* basis,
                      int T, int nb, int frame_idx, const int* offsets_host,
                      int n_off, int num_vv, int R, int S, float* pts_seq,
                      void* stream);

/* ---- a16 helpers: cross-time branch of render_rays_mono, render_ray.py:1099-1270
 * out[v] = traj(frames_a[v]) - traj(frames_b[v]) with traj(f) = sum_k coeff_k basis[f,k]
 * (scene-flow sequence :1101-1105); frames_*_host are HOST arrays, n <= 8. */
int dyn_traj_delta(const float* coeff, const float* basis, int T, int nb,
                   const int* frames_a_host, const int* frames_b_host, int n,
                   int R, int S, float* out, void* stream);
/* occ [R,S] = 1 - |w_ref - w_anchor|, occ_map [R] = 1 - |sum_s (w_ref - w_anchor)| (:1224-1257) */
int dyn_occlusion_weights(const float* w_ref, const float* w_anchor, int R, int S,
                          float* occ, float* occ_map, void* stream);

/* ---- a4-a6: Projector.compute_with_motions, projection.py:103-176 ---------
 * xyz_st [R,S,3]; xyz [V,R,S,3] or NULL (every view uses xyz_st: the static
 * branch, render_ray.py:498-500); query_cam [34]; src_rgbs [V,H,W,3]
 * channels-last in [0,1]; src_cams [V,34]; featmaps [V,C,h,w] (reference
 * layout).  Outputs rgb_feat [R,S,V,3+C], ray_diff [R,S,V,4], mask [R,S,V].
 * feat_cl_ws: workspace of V*h*w*C floats for the channels-last copy of the
 * feature maps. */
int dyn_project_gather(const float* xyz_st, const float* xyz,
                       const float* query_cam, const float* src_rgbs,
                       const float* src_cams, const float* featmaps, int V,
                       int R, int S, int H, int W, int C, int h, int w,
                       float* feat_cl_ws, float* rgb_feat, float* ray_diff,
                       float* mask, void* stream);
/* compute_projections only (projection.py:32-59): pix [V,N,2], front [V,N] u8 */
int dyn_compute_projections(const float* xyz, const float* src_cams, int V,
                            int N, float* pix, uint8_t* front, void* stream);

/* compute_angle only (projection.py:61-101): xyz_st [st_views,N,3] with st_views 1 (same reference
 * point for every view) or V; xyz [V,N,3]; ray_diff [V,N,4] = [normalize(a - b), a . b] with
 * a = normalize(c_tgt - xyz_st), b = normalize(c_src_v - xyz_v). */
int dyn_compute_angle(const float* xyz_st, int st_views, const float* xyz,
                      const float* query_cam, const float* src_cams, int V, int N,
                      float* ray_diff, void* stream);

/* ---- a7: Plucker coordinates, render_ray.py:372-396 ---------------------- */
int dyn_plucker_ref(const float* ray_o, const float* ray_d, int R, float* out6,
                    void* stream);
int dyn_plucker_src(const float* pts, const float* src_cams, int V, int R,
                    int S, float* out /* [R,S,V,6] */, void* stream);

/* ---- a8-a11: the two aggregation networks ---------------------------------
 * DynibarDynamic.forward mlp_network.py:236-316 -> raw [R,S,4].
 * ray_dir [R,3] is the NORMALISED target ray direction (render_ray.py:455). */
size_t dyn_net_workspace_bytes(int kind, int R, int S, int V);
int dyn_net_dynamic(dyn_net_t net, const float* pts, const float* rgb_feat,
                    const float* ray_dir, const float* mask, float time, int R,
                    int S, int V, float* raw, void* workspace,
                    size_t workspace_bytes, int precision, void* stream);
/* DynibarStatic.forward mlp_network.py:423-527 -> raw [R,S,4].
 * ref_rays [R,6], src_rays [R,S,V,6] are the Plucker coordinates. */
int dyn_net_static(dyn_net_t net, const float* pts, const float* ref_rays,
                   const float* src_rays, const float* rgb_feat,
                   const float* ray_diff, const float* mask, int R, int S,
                   int V, float* raw, void* workspace, size_t workspace_bytes,
                   int precision, void* stream);

/* ---- fused a4-a11 (DYN_PREC_BF16): Projector.compute_with_motions fused INTO
 * the network evaluation -- the [R,S,V,35] gather output never reaches HBM.
 * Replaces the call pairs at render_ray.py:503-521 + :538-564 (== :715-774,
 * :998-1059).  The source views arrive in two packed per-frame layouts (pack them ONCE per frame):
 *   feat_cl  = channels-last bf16 copy [V,h,w,C] of the feature maps (dyn_featmaps_channels_last):
 *              one bilinear tap of all C = 32 channels is 64 contiguous bytes;
 *   src_rgba = the source images [V,H,W,3] padded to [V,H,W,4] fp32 (dyn_rgbs_rgba): one tap is
 *              one aligned 16-byte load.
 * mask_out [R,S,V] receives the projector mask (needed by dyn_composite).  V <= 16.
 * static:  needs ray_o, ray_d [R,3] (Plucker coordinates are formed inside).
 * dynamic: pts_seq [V,R,S,3] displaced points, ray_dir [R,3] normalised. */
size_t dyn_net_fused_workspace_bytes(int kind, int R, int S, int V);
int dyn_featmaps_channels_last(const float* featmaps, void* out_bf16, int V, int C,
                               int h, int w, void* stream);
int dyn_rgbs_rgba(const float* src_rgbs, float* out_rgba, int V, int H, int W,
                  void* stream);
int dyn_net_static_fused(dyn_net_t net, const float* pts, const float* ray_o,
                         const float* ray_d, const float* query_cam,
                         const float* src_rgba, const float* src_cams,
                         const void* feat_cl, int R, int S, int V, int H,
                         int W, int C, int h, int w, float* raw,
                         float* mask_out, void* workspace,
                         size_t workspace_bytes, void* stream);
int dyn_net_dynamic_fused(dyn_net_t net, const float* pts, const float* pts_seq,
                          const float* ray_dir, const float* query_cam,
                          const float* src_rgba, const float* src_cams,
                          const void* feat_cl, float time, int R, int S, int V,
                          int H, int W, int C, int h, int w, float* raw,
                          float* mask_out, void* workspace,
                          size_t workspace_bytes, void* stream);

/* ---- a12: raw2outputs / raw2outputs_vanilla, render_ray.py:134-330 --------
 * raw_* [R,S,4]; z_vals [R,S]; mask_* [R,S,V*] as produced by
 * dyn_project_gather; a sample is "observed" when more than `min_views_*`
 * views see it (1 for the reference-time pass render_ray.py:524-529, 0 for the
 * anchor pass :1198-1200); ray mask = observed samples > 8.
 * out_rays [R,11]: rgb(3) rgb_static(3) rgb_dy(3) depth(1) mask(1, 0/1);
 * out_samples [5,R,S]: alpha_dy, weights_dy, weights_st, alpha, weights. */
int dyn_composite(const float* raw_dy, const float* raw_st,
                  const float* z_vals, const float* mask_dy, int V_dy,
                  int min_views_dy, const float* mask_st, int V_st,
                  int min_views_st, int R, int S, float* out_rays,
                  float* out_samples, void* stream);
/* out_rays [R,5]: rgb(3) depth(1) mask(1); out_samples [2,R,S]: weights, alpha */
int dyn_composite_vanilla(const float* raw, const float* z_vals,
                          const float* mask, int V, int min_views, int R,
                          int S, float* out_rays, float* out_samples,
                          void* stream);

/* ---- a13: sample_pdf + merge, render_ray.py:19-64, :790-819 ---------------
 * z_vals [R,S], weights [R,S] (coarse `weights`); u [R,Ni] uniforms or NULL
 * (det: linspace(0,1,Ni)).  z_out [R,S+Ni] sorted ascending. */
int dyn_resample(const float* z_vals, const float* weights, const float* u,
                 int R, int S, int Ni, int inv_uniform, float* z_out,
                 void* stream);

/* Training of the 2-D encoder (row f2; autograd of ResNet.forward, feature_network.py:302-311 with BasicBlock.forward
 * :68-84).  The train forward keeps every pre-norm convolution output, activation and InstanceNorm statistic in `saved`
 * (dyn_encoder_train_workspace_bytes); the backward ACCUMULATES d(loss)/d(params) into d_params (n_params floats, the
 * order of dyn_encoder_forward's `params`; the caller zeroes it) from d_coarse / d_fine [N,32,H/4,W/4] (either may be
 * NULL).  The images carry no gradient.  Every convolution is differentiated through its im2col form; `precision`
 * DYN_PREC_BF16 runs the two products per convolution on tcgen05 (bf16 operands, fp32 accumulation). */
size_t dyn_encoder_train_workspace_bytes(int N, int H, int W);
size_t dyn_encoder_backward_scratch_bytes(int N, int H, int W);
int dyn_encoder_train_forward(const float* params, size_t n_params, const float* images, int N, int H, int W,
                              float* coarse, float* fine, void* saved, size_t saved_bytes, void* stream);
int dyn_encoder_backward(const float* params, size_t n_params, const float* images, int N, int H, int W,
                         const float* d_coarse, const float* d_fine, void* saved, size_t saved_bytes,
                         void* scratch, size_t scratch_bytes, float* d_params, int precision, void* stream);

/* ---- a14: flow / expected scene flow, render_ray.py:333-358, :585-595 -----
 * weights [R,S]; pts_seq [V,R,S,3] (first n_flow views used); src_cams
 * [V,34]; uv [R,2]; coeff [R,S,3*nb]; basis [T,nb]; sf_k = 2 (mv) or 1 (mono).
 * flows [n_flow,R,2]; exp_sf [R,3]. */
int dyn_flow_sceneflow(const float* weights, const float* pts_seq,
                       const float* src_cams, const float* uv,
                       const float* coeff, const float* basis, int T, int nb,
                       int frame_idx, int sf_k, int n_flow, int R, int S,
                       float* flows, float* exp_sf, void* stream);

/* ---- f2 (first slice): backward of the two non-MLP ends of the path -------------------------
 * dyn_composite_backward: raw2outputs (render_ray.py:214-330).  g_rays [R,11] = d/d(rgb, rgb_static,
 * rgb_dy, depth, mask(ignored)), g_samples [5,R,S] = d/d(alpha_dy, weights_dy, weights_st, alpha,
 * weights) or NULL -> g_raw_dy, g_raw_st [R,S,4].  S <= 256.
 * dyn_project_gather_backward: compute_with_motions (projection.py:103-176).  g_rgb_feat [R,S,V,3+C]
 * -> g_featmaps [V,C,h,w] (reference layout; zeroed here, atomically accumulated) and / or g_xyz [V,R,S,3]
 * (either may be NULL).  xyz may be NULL (every view uses xyz_st). */
int dyn_composite_backward(const float* raw_dy, const float* raw_st, const float* z_vals,
                           const float* g_rays, const float* g_samples, int R, int S,
                           float* g_raw_dy, float* g_raw_st, void* stream);
int dyn_project_gather_backward(const float* xyz_st, const float* xyz, const float* src_rgbs,
                                const float* src_cams, const float* featmaps,
                                const float* g_rgb_feat, int V, int R, int S, int H, int W,
                                int C, int h, int w, float* g_featmaps, float* g_xyz,
                                void* stream);

/* MotionMLP training slice (ibrnet/mlp_network.py:605-618; gradients as torch.autograd would produce them
 * for MotionMLP.forward).  The forward keeps the embedding and the eight post-ReLU activations in `saved`
 * (dyn_motion_train_workspace_bytes(N) bytes, also scratch for the backward).  The backward ACCUMULATES
 * d(loss)/d(params) into d_params (flat, the n_params floats of dyn_net_create, same layout as the
 * blob given to dyn_net_create; the caller zeroes it) and writes d(loss)/d(xyzt) [N,4] unless d_xyzt is NULL.
 * fp32; split-K float atomics (not bit-reproducible between runs). */
size_t dyn_motion_train_workspace_bytes(int N);
int dyn_motion_mlp_train_forward(dyn_net_t motion, const float* xyzt, int N, float* coeff, void* saved,
                                 size_t saved_bytes, int precision, void* stream);
int dyn_motion_mlp_backward(dyn_net_t motion, const float* xyzt, const float* d_coeff, int N, void* saved,
                            size_t saved_bytes, float* d_params, float* d_xyzt, int precision, void* stream);

/* ---- f2: training step of the two aggregation networks (DynibarDynamic.forward, ibrnet/mlp_network.py:236-316;
 * DynibarStatic.forward, :423-527; gradients as torch.autograd produces them for those modules).
 * The *_train_forward calls are the fp32 forwards of dyn_net_dynamic / dyn_net_static that keep every activation in
 * `saved` (dyn_net_train_workspace_bytes bytes; R rays must fit one internal chunk: R*S*V <= 4 Mi rows).  The
 * backward reads `saved`, uses `scratch` (dyn_net_backward_scratch_bytes), ACCUMULATES d(loss)/d(params) into
 * d_params (flat, layout of the blob given to dyn_net_create; the caller zeroes it) and writes
 * d_rgb_feat [R,S,V,35] (gradient w.r.t. the gathered colours + features; NULL to skip) and, for the dynamic net,
 * d_pts [R,S,3] (through the positional encoding of ref_pts_fc; NULL to skip).  mask / ray_diff / rays / time carry
 * no gradient (the reference detaches them).  `precision`: DYN_PREC_FP32 = SIMT products; DYN_PREC_BF16 = the
 * products of the large layers on tcgen05 (bf16 operands, fp32 accumulation, fp32 master weights / gradients; the
 * net must have been created with layer images, dyn_net_create_ex pack_level >= 1); everything else stays fp32.
 * Float atomics (not bit-reproducible between runs). */
size_t dyn_net_train_workspace_bytes(int kind, int R, int S, int V);
size_t dyn_net_backward_scratch_bytes(int kind, int R, int S, int V);
int dyn_net_dynamic_train_forward(dyn_net_t net, const float* pts, const float* rgb_feat, const float* ray_dir,
                                  const float* mask, float time, int R, int S, int V, float* raw, void* saved,
                                  size_t saved_bytes, int precision, void* stream);
int dyn_net_dynamic_backward(dyn_net_t net, const float* pts, const float* mask, int R, int S, int V,
                             const float* d_raw, void* saved, size_t saved_bytes, void* scratch,
                             size_t scratch_bytes, float* d_params, float* d_rgb_feat, float* d_pts, int precision,
                             void* stream);
int dyn_net_static_train_forward(dyn_net_t net, const float* pts, const float* ref_rays, const float* src_rays,
                                 const float* rgb_feat, const float* ray_diff, const float* mask, int R, int S,
                                 int V, float* raw, void* saved, size_t saved_bytes, int precision, void* stream);
int dyn_net_static_backward(dyn_net_t net, const float* rgb_feat, const float* ray_diff, int R, int S, int V,
                            const float* d_raw, void* saved, size_t saved_bytes, void* scratch,
                            size_t scratch_bytes, float* d_params, float* d_rgb_feat, int precision, void* stream);

/* Smaller pieces of the training step:
 * dyn_composite_vanilla_backward: raw2outputs_vanilla (render_ray.py:134-211).  g_rays [R,5] = d/d(rgb, depth,
 *   mask(ignored)), g_samples [2,R,S] = d/d(weights, alpha) or NULL -> g_raw [R,S,4].  S <= 256.
 * dyn_traj_combine(_backward): compute_traj_pts and the displacements built from it (render_ray.py:361-369,
 *   :462-500, :1101-1176): out[i,p,:] = (base ? base[p,:] : 0) + sum_k coeff[p, axis*nb + k] * D[i,k]; D [n,nb]
 *   (DEVICE; rows = differences of DCT basis rows), coeff [P,3*nb], base [P,3] or NULL, out [n,P,3].  The backward
 *   writes g_coeff [P,3*nb] and / or g_base [P,3] (either may be NULL).
 * dyn_flow_backward: compute_optical_flow (render_ray.py:333-358) -> g_weights [R,S], g_pts_seq [n_flow,R,S,3]
 *   (either may be NULL).  S <= 256. */
int dyn_composite_vanilla_backward(const float* raw, const float* z_vals, const float* g_rays,
                                   const float* g_samples, int R, int S, float* g_raw, void* stream);
int dyn_traj_combine(const float* coeff, const float* D, const float* base, int n, int nb, int P, float* out,
                     void* stream);
int dyn_traj_combine_backward(const float* g_out, const float* D, int n, int nb, int P, float* g_coeff,
                              float* g_base, void* stream);
int dyn_flow_backward(const float* weights, const float* pts_seq, const float* src_cams, const float* g_flows,
                      int n_flow, int R, int S, float* g_weights, float* g_pts_seq, void* stream);

/* ---- training objective: train.py:300-458 (the loss of one training step), the static-bootstrap loss of
 * train.py:187-196 and eff_distloss_native (mip-NeRF 360 distortion, prefix-sum form), with the criteria of
 * ibrnet/criterion.py.  One warp per ray; every per-ray quantity is evaluated in fp64.
 *
 * `in` describes the tensors (all [R]-leading rows dense fp32; masks as 0/1 floats):
 *   outputs_coarse_ref      rgb, rgb_dy, rgb_static [R,3]; depth, mask [R]; weights, weights_dy, weights_st,
 *                           s_vals [R,S]; render_flows [F,R,2]
 *   outputs_coarse_ref_dy   ref_dy_rgb [R,3], ref_dy_mask [R]
 *   outputs_coarse_anchor   a_rgb [R,3], a_mask, a_occ_map [R], occ_weights [R,S],
 *                           pts_traj_ref, pts_traj_anchor [K,R,S,3], sf_seq [T,R,S,3]
 *   outputs_coarse_anchor_dy a_dy_rgb [R,3], a_dy_mask, a_dy_occ_map [R]
 *   outputs_coarse_st       st_rgb [R,3]
 *   ray_batch               gt_rgb [R,3], disp, motion_mask, static_mask [R], flows [F,R,2], flow_masks [F,R,1]
 *   eff_distloss_native     dist_mid, dist_interval [R,S] with weights [R,S] = w; when both are NULL the
 *                           distortion term reads weights[:, :S-1], mid(s_vals) and diff(s_vals) instead.
 * Only the tensors of the enabled `terms` (DYN_OBJ_* bits) are read; the others may be NULL.
 *
 * dyn_objective_sums writes the DYN_OBJ_NSUMS fp64 sums of the batch (numerators, denominators and the ray /
 * element counts of the means; slots DYN_OBJ_SUM_*), reduced per block in warp order and across blocks in block
 * order: no float atomics, bit-identical between runs.  Sums of disjoint ray batches add up to the sums of their
 * union, so sharded callers all-reduce this vector (SUM) before dyn_objective_finalize.
 * dyn_objective_finalize turns a sums vector into loss [1] and the DYN_OBJ_NTERMS term values (fp32; order
 * rgb, flow, disp, distortion, entropy, static, cycle, reg) and `scales` [DYN_OBJ_NSUMS] fp64: d loss / d each
 * numerator.  coef_host [DYN_OBJ_NCOEF] (HOST): dynamic-rgb factor 1/10^divisor, disp, flow, cycle, reg,
 * entropy and distortion weights.
 * dyn_objective_backward writes every non-NULL gradient of `grad` in full from the upstream gradients g_loss [1]
 * and g_terms [DYN_OBJ_NTERMS] (device; either may be NULL = 0) and the scales of the finalize step.
 * One launch each; nothing synchronises. */
#define DYN_OBJ_RGB 0x001            /* Charbonnier of ref.rgb under ref.mask (train.py:304) */
#define DYN_OBJ_TEMPORAL 0x002       /* temporal Charbonnier of anchor.rgb (:305-307) */
#define DYN_OBJ_DYREGION 0x004       /* Charbonnier of ref.rgb_dy under mask * motion_mask (:309-316) */
#define DYN_OBJ_DYNAMIC 0x008        /* ref_dy.rgb and anchor_dy.rgb under motion_mask, / 10^divisor (:318-329) */
#define DYN_OBJ_DISP 0x010           /* disparity L1 (:330-343) */
#define DYN_OBJ_FLOW 0x020           /* flow L1 (:344-352) */
#define DYN_OBJ_CYCLE 0x040          /* trajectory cycle L1 (:353-371) */
#define DYN_OBJ_REG 0x080            /* scene-flow regularisers (:373-397) */
#define DYN_OBJ_ENTROPY 0x100        /* weight-ratio entropy (:399-413) */
#define DYN_OBJ_DISTORTION 0x200     /* eff_distloss_native (:415-423) */
#define DYN_OBJ_STATIC 0x400         /* static Charbonnier of ref.rgb_static (:425-435) */
#define DYN_OBJ_STATIC_EXTRA 0x800   /* divisor > 4: zero dynamic weight where ratio < 0.1 (:437-445) */
#define DYN_OBJ_BOOTSTRAP 0x1000     /* static bootstrap, Charbonnier of st.rgb (:187-196) */
#define DYN_OBJ_NSUMS 32
#define DYN_OBJ_NTERMS 8
#define DYN_OBJ_NCOEF 7

typedef struct dyn_objective_in {
  int R, S, K, T, F; /* rays, samples, trajectory views, sf_seq steps, flow views */
  const float *rgb, *rgb_dy, *rgb_static, *depth, *mask, *weights, *weights_dy, *weights_st, *s_vals,
      *render_flows;
  const float *ref_dy_rgb, *ref_dy_mask;
  const float *a_rgb, *a_mask, *a_occ_map, *occ_weights, *pts_traj_ref, *pts_traj_anchor, *sf_seq;
  const float *a_dy_rgb, *a_dy_mask, *a_dy_occ_map;
  const float* st_rgb;
  const float *gt_rgb, *disp, *motion_mask, *static_mask, *flows, *flow_masks;
  const float *dist_mid, *dist_interval;
} dyn_objective_in;

typedef struct dyn_objective_grad { /* same shapes as the inputs of the same names */
  float *rgb, *rgb_dy, *rgb_static, *depth, *weights, *weights_dy, *weights_st, *render_flows;
  float* ref_dy_rgb;
  float *a_rgb, *pts_traj_ref, *pts_traj_anchor, *sf_seq;
  float* a_dy_rgb;
  float* st_rgb;
} dyn_objective_grad;

size_t dyn_objective_workspace_bytes(int R);
int dyn_objective_sums(const dyn_objective_in* in, int terms, double* sums, void* workspace,
                       size_t workspace_bytes, void* stream);
int dyn_objective_finalize(const double* sums, int terms, const double* coef_host, float* loss, float* term_values,
                           double* scales, void* stream);
int dyn_objective_backward(const dyn_objective_in* in, int terms, const double* scales, const float* g_loss,
                           const float* g_terms, const dyn_objective_grad* grad, void* stream);

/* Unit-test hooks of the tensor-core training products (csrc/train_tc.cu; bf16 operands, fp32 accumulation):
 * dyn_debug_tc_grad_w: dW[out,width] += dz[rows,out]^T (x[rows,width] * kscale[rows] or 1); out, width <= 256.
 * dyn_debug_tc_grad_in: din[rows,width] = dz[rows,out] W[out, 0:width] (W row-major with ldw columns). */
int dyn_debug_tc_grad_w(const float* dz, int lddz, int out, int rows, const float* x, int ldx, int width,
                        const float* kscale, float* dW, int ldw, void* stream);
int dyn_debug_tc_grad_in(const float* dz, int lddz, int out, int rows, const float* W, int ldw, int width,
                         float* din, int ldd, void* scratch, size_t scratch_bytes, void* stream);
size_t dyn_debug_tc_grad_in_scratch_bytes(void);

/* ---- f1: 2-D feature encoder, ResNet.forward as the reference runs it (feature_network.py:302-311) ----
 * conv 7x7 stride 2 (reflect) -> InstanceNorm -> ReLU -> layer1 (3 BasicBlocks, the first with stride 2)
 * -> 1x1 conv -> coarse (channels 0..31) | fine (channels 32..63).  images [N,3,H,W] fp32;
 * coarse, fine [N,32,H/4,W/4].  `params` = the executed parameters in state_dict order
 * (dynibar_b200/feature_network.py: _EXECUTED), dyn_encoder_param_count() floats. */
size_t dyn_encoder_param_count(void);
size_t dyn_encoder_workspace_bytes(int N, int H, int W);
int dyn_encoder_forward(const float* params, size_t n_params, const float* images,
                        int N, int H, int W, float* coarse, float* fine,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- unit-test hook: the fused per-point stage (geometry_fc -> ray transformer
 * -> heads; mlp_network.py:283-315 / :496-506) on caller-provided pooled
 * features G [R*S, 272] (257 used) and nvalid [R*S].  Outputs g2 [R*S,128] (plain
 * fp32 rows; the Q, K, V, O arguments are ignored: those intermediates live in
 * the kernels' internal tile-image scratch); dynamic net: out_a = raw [R*S,4]; static net:
 * out_a = per-point part of rgb_fc.0 [R*S,128], out_b = masked sigma [R*S].
 * posenc_ws: S*128 floats of scratch. */
int dyn_debug_point_chain(dyn_net_t net, const float* G, const float* nvalid,
                          const float* pts, const float* ray_dir, int R, int S,
                          float* g2, float* Q, float* K, float* V, float* O,
                          float* out_a, float* out_b, float* posenc_ws,
                          void* stream);

/* ---- unit-test hook (HOST only, no GPU needed): pack one nn.Linear [N, Kw] into the bf16
 * UMMA weight image the fused kernels stream (dynibar_b200/csrc/fused_engine.cuh:
 * append_layer).  colmap[Kpad] maps operand column -> weight column, -1 = zero,
 * -2 / -3 = hi / lo bf16 halves of the folded bias; `scale` multiplies weights and
 * bias.  Chunks of `stage_bytes`; element (n, k) of a chunk that starts at k0 sits at
 * byte ((k-k0)/8)*(Npad*16) + (n/8)*128 + (n%8)*16 + ((k-k0)%8)*2 of that chunk.
 * Writes the image into out_img (out_bytes capacity), its size into *img_bytes and the
 * number of chunks into *nchunks. */
int dyn_debug_pack_layer(const float* W, const float* bias, int N, int Kw, int Npad,
                         int Kpad, const int* colmap, float scale, int stage_bytes,
                         void* out_img, size_t out_bytes, size_t* img_bytes,
                         int* nchunks);
/* byte offset of (row, 8-column group) in a bf16 tile image with `kgroups` groups per
 * 128-row tile: the layout activations use between the fused kernels. */
size_t dyn_debug_tile_image_off(long long row, int kgroup, int kgroups);

/* measurement hook: which kernel runs the fused per-view stage.  -1 (the initial value) = the library's
 * kernel (csrc/view_twin3.cu).  The comparison variants 0 (round-1 twin-warp kernel), 1 (quad schedule) and
 * 2 (sub-round pipelined twin kernel without elected arrive) were removed: with any value other than -1 every
 * fused per-view call (dyn_net_static_fused / dyn_net_dynamic_fused) fails with DYN_E_INVALID and
 * dyn_last_error() names the variant, so a measurement asking for one cannot time the default instead. */
void dyn_debug_set_view_kernel(int which);

/* profiling hook: when set, block 0 of the fused static per-view kernel writes clock64()
 * phase timestamps ([2 twins][64]) into dev_buf (profiles/scripts/prof_phases.py). */
void dyn_debug_set_view_timestamps(long long* dev_buf);

/* ---- building block: one nn.Linear on the tensor cores -----------------------
 * Y[M,N] = act(X[M,K] W[N,K]^T + b) with bf16 operands / fp32 accumulation
 * (tcgen05).  act: 0 none, 1 ELU, 2 ReLU, 3 sigmoid.  N <= 256.  packed_ws must
 * hold dyn_linear_tc_packed_bytes(N, K) bytes (bf16 UMMA image of W).  This is
 * the kernel behind every nn.Linear of mlp_network.py in DYN_PREC_BF16 mode;
 * exported for unit testing. */
size_t dyn_linear_tc_packed_bytes(int N, int K);
int dyn_linear_tc(const float* X, int ldx, const float* W, const float* b, int M,
                  int N, int K, int act, float* Y, int ldy, void* packed_ws,
                  size_t packed_ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DYNIBAR_B200_H_ */
