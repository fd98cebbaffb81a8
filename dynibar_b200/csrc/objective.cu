// Training objective of one DynIBaR step (train.py:300-458), the static-bootstrap loss (train.py:187-196) and
// eff_distloss_native, forward and analytic backward.
//
//   objective_sums_kernel      one warp per ray: the ray's contribution to every numerator, denominator and count
//                              of the objective (fp64), reduced in a fixed order -- lanes by a butterfly, warps in
//                              warp order, blocks in block order by the last block to finish (integer ticket).
//   objective_finalize_kernel  sums -> loss, the eight logged terms and d loss / d numerator (one thread).
//   objective_backward_kernel  one warp per ray: every input gradient, from the upstream gradients and the scales.
//
// Every loss of the objective is a ratio N / D whose denominator D holds only detached quantities (masks,
// occlusion weights, counts), so d loss / d x = (coefficient / D) * d N / d x: the backward needs the finalized
// scales and the ray's own inputs, nothing else.  With the sums all-reduced over ranks each rank's loss is the
// full-batch loss and its gradients are its rays' share of the full-batch gradient.
//
// Thresholds that the reference applies to fp32 tensors (clamp(depth, 1e-2)) are applied in fp32 here too, so a
// value sitting exactly on one takes the same branch as in torch.
#include "common.cuh"

namespace dyn {

namespace {

constexpr int kWarps = 8;  // rays per block

enum Slot {
  S_RGB_N, S_RGB_D,     // ref.rgb Charbonnier; D = sum ref.mask (also the disparity denominator)
  S_TMP_N, S_TMP_D,     // anchor.rgb temporal Charbonnier
  S_DYR_N, S_DYR_D,     // ref.rgb_dy under mask * motion_mask
  S_RDY_N, S_RDY_D,     // ref_dy.rgb under ref_dy.mask * motion_mask
  S_ADY_N, S_ADY_D,     // anchor_dy.rgb temporal, motion_mask
  S_DISP_N,
  S_FLOW_N, S_FLOW_D,
  S_CYC_N, S_CYC_D,
  S_SF_ABS, S_SF_T2, S_SF_DS,  // sum |sf|, sum (sf_t - sf_t+1)^2, sum |sf_s+1 - sf_s|
  S_ENT, S_DIST,
  S_ST_N, S_ST_D,       // ref.rgb_static under (1 - static_mask) * mask * (1 - ratio)
  S_X_N, S_X_D,         // divisor > 4 term
  S_BOOT_N, S_BOOT_D,   // static bootstrap
  S_RAYS, S_SF_CNT, S_SF_T_CNT, S_SF_S_CNT,
  S_NUM
};
static_assert(S_NUM <= DYN_OBJ_NSUMS, "sums vector too short");

// term (index into the DYN_OBJ_NTERMS values: rgb, flow, disp, distortion, entropy, static, cycle, reg) that each
// numerator slot belongs to; -1 for denominators and counts
__constant__ signed char kTermOf[DYN_OBJ_NSUMS] = {
    0, -1, 0, -1, 0, -1, 0, -1, 0, -1,  // rgb terms
    2,                                  // disp
    1, -1,                              // flow
    6, -1,                              // cycle
    7, 7, 7,                            // reg
    4, 3,                               // entropy, distortion
    5, -1, 5, -1, 5, -1,                // static, extra, bootstrap
    -1, -1, -1, -1, -1, -1};

constexpr double kCharbEps2 = 1e-6;  // criterion.py:19, EPSILON**2
constexpr double kLogEps = 1e-9;     // train.py:410-411
constexpr float kClampRatio = 1e-9f;  // train.py:406-408 (fp32 tensor)
constexpr float kClampDepth = 1e-2f;  // train.py:332-334 (fp32 tensor)

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_incl_scan_d(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
__device__ __forceinline__ double sgn(double x) { return (double)((x > 0.0) - (x < 0.0)); }  // abs'(0) = 0
__device__ __forceinline__ double charb(float x, float y) {
  const double d = (double)x - (double)y;
  return sqrt(d * d + kCharbEps2);
}
__device__ __forceinline__ double charb_grad(float x, float y) {
  const double d = (double)x - (double)y;
  return d / sqrt(d * d + kCharbEps2);
}
__device__ __forceinline__ double ld(const float* p, long long i) { return (double)p[i]; }

// per-ray quantities both kernels need
struct RayCtx {
  double m, motion, wd, ws, ratio, clampsum_ok, mask_s;
};

__device__ RayCtx ray_ctx(const dyn_objective_in& in, int terms, int r, int lane) {
  RayCtx c{};
  c.m = in.mask ? ld(in.mask, r) : 0.0;
  c.motion = in.motion_mask ? ld(in.motion_mask, r) : 0.0;
  if (terms & (DYN_OBJ_ENTROPY | DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA)) {
    double wd = 0.0, ws = 0.0;
    for (int s = lane; s < in.S; s += 32) {
      wd += ld(in.weights_dy, (long long)r * in.S + s);
      ws += ld(in.weights_st, (long long)r * in.S + s);
    }
    c.wd = warp_sum_d(wd);
    c.ws = warp_sum_d(ws);
    const double sum = c.wd + c.ws;
    c.clampsum_ok = sum >= (double)kClampRatio ? 1.0 : 0.0;  // clamp passes the gradient where x >= min
    c.ratio = c.wd / fmax(sum, (double)kClampRatio);
  }
  if (terms & (DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA))
    c.mask_s = (1.0 - ld(in.static_mask, r)) * c.m * (1.0 - c.ratio);  // (1 - ratio) detached (train.py:428)
  return c;
}

// distortion samples of ray r: weight, midpoint, interval of sample i < n
__device__ __forceinline__ void dist_sample(const dyn_objective_in& in, int r, int i, double& w, double& mid,
                                            double& iv) {
  const long long o = (long long)r * in.S + i;
  w = ld(in.weights, o);
  if (in.dist_mid) {
    mid = ld(in.dist_mid, o);
    iv = ld(in.dist_interval, o);
  } else {
    const double a = ld(in.s_vals, o), b = ld(in.s_vals, o + 1);
    mid = (b + a) * 0.5;
    iv = b - a;
  }
}
__device__ __forceinline__ int dist_n(const dyn_objective_in& in) { return in.dist_mid ? in.S : in.S - 1; }

__global__ void __launch_bounds__(kWarps * 32)
objective_sums_kernel(const dyn_objective_in in, int terms, double* __restrict__ part,
                      unsigned int* __restrict__ ticket, double* __restrict__ sums) {
  __shared__ double sh[kWarps][S_NUM];
  __shared__ bool is_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * kWarps + warp;
  for (int i = lane; i < S_NUM; i += 32) sh[warp][i] = 0.0;
  __syncwarp();
  if (r < in.R) {
    const int S = in.S;
    const long long RS = (long long)in.R * S;
    // warp-summed lane partials / ray-uniform values
    auto put = [&](int slot, double v) {
      v = warp_sum_d(v);
      if (lane == 0) sh[warp][slot] = v;
    };
    auto put1 = [&](int slot, double v) {
      if (lane == 0) sh[warp][slot] = v;
    };
    const RayCtx c = ray_ctx(in, terms, r, lane);
    const int ch = lane < 3 ? lane : 0;
    const long long rc = (long long)r * 3 + ch;
    const double on3 = lane < 3 ? 1.0 : 0.0;
    if (terms & DYN_OBJ_RGB) {
      put(S_RGB_N, on3 * c.m * charb(in.rgb[rc], in.gt_rgb[rc]));
      put1(S_RGB_D, c.m);
    }
    if (terms & DYN_OBJ_TEMPORAL) {
      const double w = ld(in.a_mask, r) * ld(in.a_occ_map, r);
      put(S_TMP_N, on3 * w * charb(in.a_rgb[rc], in.gt_rgb[rc]));
      put1(S_TMP_D, w);
    }
    if (terms & DYN_OBJ_DYREGION) {
      const double w = c.m * c.motion;
      put(S_DYR_N, on3 * w * charb(in.rgb_dy[rc], in.gt_rgb[rc]));
      put1(S_DYR_D, w);
    }
    if (terms & DYN_OBJ_DYNAMIC) {
      const double w = ld(in.ref_dy_mask, r) * c.motion;
      put(S_RDY_N, on3 * w * charb(in.ref_dy_rgb[rc], in.gt_rgb[rc]));
      put1(S_RDY_D, w);
      const double wa = ld(in.a_dy_mask, r) * c.motion * ld(in.a_dy_occ_map, r);
      put(S_ADY_N, on3 * wa * charb(in.a_dy_rgb[rc], in.gt_rgb[rc]));
      put1(S_ADY_D, wa);
    }
    if (terms & DYN_OBJ_DISP) {
      const float cl = fmaxf(in.depth[r], kClampDepth);
      put1(S_DISP_N, fabs(1.0 / (double)cl - ld(in.disp, r)) * c.m);
      put1(S_RGB_D, c.m);
    }
    if (terms & DYN_OBJ_FLOW) {
      double n = 0.0, d = 0.0;
      for (int j = lane; j < 2 * in.F; j += 32) {
        const int f = j >> 1;
        const double fm = c.m * ld(in.flow_masks, (long long)f * in.R + r);
        const long long o = ((long long)f * in.R + r) * 2 + (j & 1);
        n += fabs(ld(in.render_flows, o) - ld(in.flows, o)) * fm;
        d += fm;
      }
      put(S_FLOW_N, n);
      put(S_FLOW_D, d);
    }
    if (terms & DYN_OBJ_CYCLE) {
      double n = 0.0, d = 0.0;
      for (int k = 0; k < in.K; ++k) {
        const long long base = ((long long)k * in.R + r) * S * 3;
        for (int e = lane; e < S * 3; e += 32) {
          const double occ = ld(in.occ_weights, (long long)r * S + e / 3);
          n += fabs(ld(in.pts_traj_ref, base + e) - ld(in.pts_traj_anchor, base + e)) * occ;
          d += occ;
        }
      }
      put(S_CYC_N, n);
      put(S_CYC_D, d);
    }
    if (terms & DYN_OBJ_REG) {
      double a = 0.0, t2 = 0.0, ds = 0.0;
      for (int t = 0; t < in.T; ++t) {
        const long long base = ((long long)t * in.R + r) * S * 3;
        for (int e = lane; e < S * 3; e += 32) {
          const double x = ld(in.sf_seq, base + e);
          a += fabs(x);
          if (t + 1 < in.T) {
            const double y = x - ld(in.sf_seq, base + RS * 3 + e);
            t2 += y * y;
          }
          if (e + 3 < S * 3) ds += fabs(ld(in.sf_seq, base + e + 3) - x);
        }
      }
      put(S_SF_ABS, a);
      put(S_SF_T2, t2);
      put(S_SF_DS, ds);
      put1(S_SF_CNT, (double)in.T * S * 3);
      put1(S_SF_T_CNT, (double)(in.T - 1) * S * 3);
      put1(S_SF_S_CNT, (double)in.T * (S - 1) * 3);
    }
    if (terms & DYN_OBJ_ENTROPY) {
      const double q = c.ratio;
      put1(S_ENT, -(q * log(q + kLogEps) + (1.0 - q) * log(1.0 - q + kLogEps)));
    }
    if (terms & DYN_OBJ_DISTORTION) {
      // (1/3) sum delta w^2 + 2 sum_i (w_i m_i W_{i-1} - w_i WM_{i-1}), W / WM inclusive prefix sums of w / w m
      const int n = dist_n(in);
      double acc = 0.0, cw = 0.0, cwm = 0.0;  // running sums of the strides before this one
      for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        double w = 0.0, mid = 0.0, iv = 0.0;
        if (i < n) dist_sample(in, r, i, w, mid, iv);
        const double W = warp_incl_scan_d(w, lane), WM = warp_incl_scan_d(w * mid, lane);
        const double Wex = cw + W - w, WMex = cwm + WM - w * mid;
        acc += iv * w * w * (1.0 / 3.0) + 2.0 * (w * mid * Wex - w * WMex);
        cw += __shfl_sync(0xffffffffu, W, 31);
        cwm += __shfl_sync(0xffffffffu, WM, 31);
      }
      put(S_DIST, acc);
    }
    if (terms & DYN_OBJ_STATIC) {
      put(S_ST_N, on3 * c.mask_s * charb(in.rgb_static[rc], in.gt_rgb[rc]));
      put1(S_ST_D, c.mask_s);
    }
    if (terms & DYN_OBJ_STATIC_EXTRA) {
      const double m2 = c.mask_s * (c.ratio < 0.1 ? 1.0 : 0.0);
      put1(S_X_N, fabs(c.wd * m2));
      put1(S_X_D, m2 + 1e-8);  // the 1e-8 sits inside the sum (train.py:444)
    }
    if (terms & DYN_OBJ_BOOTSTRAP) {
      const double w = (1.0 - ld(in.static_mask, r)) * c.m;
      put(S_BOOT_N, on3 * w * charb(in.st_rgb[rc], in.gt_rgb[rc]));
      put1(S_BOOT_D, w);
    }
    put1(S_RAYS, 1.0);
  }
  __syncthreads();
  if (threadIdx.x < S_NUM) {
    double v = 0.0;
    for (int w = 0; w < kWarps; ++w) v += sh[w][threadIdx.x];
    part[(long long)blockIdx.x * S_NUM + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x < DYN_OBJ_NSUMS) {
    double v = 0.0;
    if (threadIdx.x < S_NUM) {
      const volatile double* p = part;
      for (unsigned b = 0; b < gridDim.x; ++b) v += p[(long long)b * S_NUM + threadIdx.x];
    }
    sums[threadIdx.x] = v;
  }
  if (threadIdx.x == 0) *ticket = 0u;
}

struct Coef {
  double c[DYN_OBJ_NCOEF];
};

__global__ void objective_finalize_kernel(const double* __restrict__ sums, int terms, Coef k, float* __restrict__ loss,
                                          float* __restrict__ vals, double* __restrict__ scales) {
  if (threadIdx.x != 0) return;
  double s[S_NUM], sc[DYN_OBJ_NSUMS], t[DYN_OBJ_NTERMS];
  for (int i = 0; i < S_NUM; ++i) s[i] = sums[i];
  for (int i = 0; i < DYN_OBJ_NSUMS; ++i) sc[i] = 0.0;
  for (int i = 0; i < DYN_OBJ_NTERMS; ++i) t[i] = 0.0;
  const double c_dyn = k.c[0], c_disp = k.c[1], c_flow = k.c[2], c_cyc = k.c[3], c_reg = k.c[4], c_ent = k.c[5],
               c_dist = k.c[6];
  // rgb (utils.py:32-39: sum(mask) * 3 + 1e-6; criterion.py:55: 3 * sum(w) + 1e-8)
  if (terms & DYN_OBJ_RGB) sc[S_RGB_N] = 1.0 / (3.0 * s[S_RGB_D] + 1e-6);
  if (terms & DYN_OBJ_TEMPORAL) sc[S_TMP_N] = 1.0 / (3.0 * s[S_TMP_D] + 1e-8);
  if (terms & DYN_OBJ_DYREGION) sc[S_DYR_N] = 1.0 / (3.0 * s[S_DYR_D] + 1e-6);
  if (terms & DYN_OBJ_DYNAMIC) {
    sc[S_RDY_N] = c_dyn / (3.0 * s[S_RDY_D] + 1e-6);
    sc[S_ADY_N] = c_dyn / (3.0 * s[S_ADY_D] + 1e-8);
  }
  if (terms & DYN_OBJ_DISP) sc[S_DISP_N] = c_disp / (s[S_RGB_D] + 1e-8);
  if (terms & DYN_OBJ_FLOW) sc[S_FLOW_N] = c_flow / (s[S_FLOW_D] + 1e-8);
  if (terms & DYN_OBJ_CYCLE) sc[S_CYC_N] = c_cyc / (s[S_CYC_D] + 1e-8);
  if (terms & DYN_OBJ_REG) {  // torch.mean: sum / count
    sc[S_SF_ABS] = c_reg / s[S_SF_CNT];
    sc[S_SF_T2] = c_reg * 0.5 / s[S_SF_T_CNT];
    sc[S_SF_DS] = c_reg / s[S_SF_S_CNT];
  }
  if (terms & DYN_OBJ_ENTROPY) sc[S_ENT] = c_ent / s[S_RAYS];
  if (terms & DYN_OBJ_DISTORTION) sc[S_DIST] = c_dist / s[S_RAYS];
  if (terms & DYN_OBJ_STATIC) sc[S_ST_N] = 1.0 / (3.0 * s[S_ST_D] + 1e-6);
  if (terms & DYN_OBJ_STATIC_EXTRA) sc[S_X_N] = 0.1 / s[S_X_D];
  if (terms & DYN_OBJ_BOOTSTRAP) sc[S_BOOT_N] = 1.0 / (3.0 * s[S_BOOT_D] + 1e-6);
  double total = 0.0;
  for (int i = 0; i < S_NUM; ++i) {
    if (kTermOf[i] < 0 || sc[i] == 0.0) continue;
    t[kTermOf[i]] += s[i] * sc[i];
  }
  for (int i = 0; i < DYN_OBJ_NTERMS; ++i) total += t[i];
  *loss = (float)total;
  for (int i = 0; i < DYN_OBJ_NTERMS; ++i) vals[i] = (float)t[i];
  for (int i = 0; i < DYN_OBJ_NSUMS; ++i) scales[i] = sc[i];
}

__global__ void __launch_bounds__(kWarps * 32)
objective_backward_kernel(const dyn_objective_in in, int terms, const double* __restrict__ scales,
                          const float* __restrict__ g_loss, const float* __restrict__ g_terms,
                          const dyn_objective_grad g) {
  __shared__ double gs[DYN_OBJ_NSUMS];  // d (upstream . outputs) / d numerator
  if (threadIdx.x < DYN_OBJ_NSUMS) {
    const int term = kTermOf[threadIdx.x];
    double up = g_loss ? (double)g_loss[0] : 0.0;
    if (g_terms && term >= 0) up += (double)g_terms[term];
    gs[threadIdx.x] = term >= 0 ? up * scales[threadIdx.x] : 0.0;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * kWarps + warp;
  if (r >= in.R) return;
  const int S = in.S;
  const long long RS = (long long)in.R * S;
  const RayCtx c = ray_ctx(in, terms, r, lane);
  // [R,3] colour gradients: lanes 0..2
  auto rgb_grad = [&](float* out, const float* x, int term, int slot, double w) {
    if (!out || lane >= 3) return;
    const long long o = (long long)r * 3 + lane;
    out[o] = (terms & term) ? (float)(gs[slot] * w * charb_grad(x[o], in.gt_rgb[o])) : 0.f;
  };
  rgb_grad(g.rgb, in.rgb, DYN_OBJ_RGB, S_RGB_N, c.m);
  if (g.a_rgb) rgb_grad(g.a_rgb, in.a_rgb, DYN_OBJ_TEMPORAL, S_TMP_N,
                        (terms & DYN_OBJ_TEMPORAL) ? ld(in.a_mask, r) * ld(in.a_occ_map, r) : 0.0);
  rgb_grad(g.rgb_dy, in.rgb_dy, DYN_OBJ_DYREGION, S_DYR_N, c.m * c.motion);
  if (g.ref_dy_rgb) rgb_grad(g.ref_dy_rgb, in.ref_dy_rgb, DYN_OBJ_DYNAMIC, S_RDY_N,
                             (terms & DYN_OBJ_DYNAMIC) ? ld(in.ref_dy_mask, r) * c.motion : 0.0);
  if (g.a_dy_rgb) rgb_grad(g.a_dy_rgb, in.a_dy_rgb, DYN_OBJ_DYNAMIC, S_ADY_N,
                           (terms & DYN_OBJ_DYNAMIC) ? ld(in.a_dy_mask, r) * c.motion * ld(in.a_dy_occ_map, r) : 0.0);
  rgb_grad(g.rgb_static, in.rgb_static, DYN_OBJ_STATIC, S_ST_N, c.mask_s);
  if (g.st_rgb) rgb_grad(g.st_rgb, in.st_rgb, DYN_OBJ_BOOTSTRAP, S_BOOT_N,
                         (terms & DYN_OBJ_BOOTSTRAP) ? (1.0 - ld(in.static_mask, r)) * c.m : 0.0);
  if (g.depth && lane == 0) {
    double v = 0.0;
    if (terms & DYN_OBJ_DISP) {
      const float dep = in.depth[r];
      const float cl = fmaxf(dep, kClampDepth);
      const double e = 1.0 / (double)cl - ld(in.disp, r);
      v = dep >= kClampDepth ? gs[S_DISP_N] * c.m * sgn(e) * (-1.0 / ((double)cl * (double)cl)) : 0.0;
    }
    g.depth[r] = (float)v;
  }
  if (g.render_flows) {
    for (int j = lane; j < 2 * in.F; j += 32) {
      const int f = j >> 1;
      const long long o = ((long long)f * in.R + r) * 2 + (j & 1);
      double v = 0.0;
      if (terms & DYN_OBJ_FLOW) {
        const double fm = c.m * ld(in.flow_masks, (long long)f * in.R + r);
        v = gs[S_FLOW_N] * fm * sgn(ld(in.render_flows, o) - ld(in.flows, o));
      }
      g.render_flows[o] = (float)v;
    }
  }
  if (g.pts_traj_ref || g.pts_traj_anchor) {
    for (int k = 0; k < in.K; ++k) {
      const long long base = ((long long)k * in.R + r) * S * 3;
      for (int e = lane; e < S * 3; e += 32) {
        double v = 0.0;
        if (terms & DYN_OBJ_CYCLE) {
          const double occ = ld(in.occ_weights, (long long)r * S + e / 3);
          v = gs[S_CYC_N] * occ * sgn(ld(in.pts_traj_ref, base + e) - ld(in.pts_traj_anchor, base + e));
        }
        if (g.pts_traj_ref) g.pts_traj_ref[base + e] = (float)v;
        if (g.pts_traj_anchor) g.pts_traj_anchor[base + e] = (float)(-v);
      }
    }
  }
  if (g.sf_seq) {
    for (int t = 0; t < in.T; ++t) {
      const long long base = ((long long)t * in.R + r) * S * 3;
      for (int e = lane; e < S * 3; e += 32) {
        double v = 0.0;
        if (terms & DYN_OBJ_REG) {
          const double x = ld(in.sf_seq, base + e);
          v = gs[S_SF_ABS] * sgn(x);
          double dt = 0.0;  // d/dx sum_t (sf_t - sf_t+1)^2
          if (t + 1 < in.T) dt += 2.0 * (x - ld(in.sf_seq, base + RS * 3 + e));
          if (t > 0) dt -= 2.0 * (ld(in.sf_seq, base - RS * 3 + e) - x);
          v += gs[S_SF_T2] * dt;
          double dsp = 0.0;  // d/dx sum_s |sf_s+1 - sf_s|
          if (e + 3 < S * 3) dsp -= sgn(ld(in.sf_seq, base + e + 3) - x);
          if (e >= 3) dsp += sgn(x - ld(in.sf_seq, base + e - 3));
          v += gs[S_SF_DS] * dsp;
        }
        g.sf_seq[base + e] = (float)v;
      }
    }
  }
  if (g.weights_dy || g.weights_st) {
    double gwd = 0.0, gws = 0.0;  // d / d (sum_s weights_dy), d / d (sum_s weights_st)
    if (terms & DYN_OBJ_ENTROPY) {
      const double q = c.ratio;
      const double de = -(log(q + kLogEps) + q / (q + kLogEps) - log(1.0 - q + kLogEps) -
                          (1.0 - q) / (1.0 - q + kLogEps));
      const double den = fmax(c.wd + c.ws, (double)kClampRatio);
      const double gq = gs[S_ENT] * de;
      gwd += gq * (1.0 / den - c.clampsum_ok * c.wd / (den * den));
      gws += gq * (-c.clampsum_ok * c.wd / (den * den));
    }
    if (terms & DYN_OBJ_STATIC_EXTRA) {
      const double m2 = c.mask_s * (c.ratio < 0.1 ? 1.0 : 0.0);
      gwd += gs[S_X_N] * sgn(c.wd * m2) * m2;
    }
    for (int s = lane; s < S; s += 32) {
      if (g.weights_dy) g.weights_dy[(long long)r * S + s] = (float)gwd;
      if (g.weights_st) g.weights_st[(long long)r * S + s] = (float)gws;
    }
  }
  if (g.weights) {
    const int n = (terms & DYN_OBJ_DISTORTION) ? dist_n(in) : 0;
    double tw = 0.0, twm = 0.0;  // totals of w and w m over the ray
    for (int i = lane; i < n; i += 32) {
      double w, mid, iv;
      dist_sample(in, r, i, w, mid, iv);
      tw += w;
      twm += w * mid;
    }
    tw = warp_sum_d(tw);
    twm = warp_sum_d(twm);
    // d/dw_j = (2/3) delta_j w_j + 2 (m_j W_{<j} - WM_{<j} + WM_{>j} - m_j W_{>j})
    double cw = 0.0, cwm = 0.0;
    for (int i0 = 0; i0 < S; i0 += 32) {
      const int i = i0 + lane;
      double w = 0.0, mid = 0.0, iv = 0.0;
      if (i < n) dist_sample(in, r, i, w, mid, iv);
      const double W = warp_incl_scan_d(w, lane), WM = warp_incl_scan_d(w * mid, lane);
      const double Wlo = cw + W - w, WMlo = cwm + WM - w * mid;  // sums over i' < i
      const double Whi = tw - (cw + W), WMhi = twm - (cwm + WM);  // sums over i' > i
      cw += __shfl_sync(0xffffffffu, W, 31);
      cwm += __shfl_sync(0xffffffffu, WM, 31);
      if (i < S) {
        const double v = i < n ? gs[S_DIST] * ((2.0 / 3.0) * iv * w + 2.0 * (mid * Wlo - WMlo + WMhi - mid * Whi))
                               : 0.0;
        g.weights[(long long)r * S + i] = (float)v;
      }
    }
  }
}

// names the first tensor an enabled term needs but did not get
const char* missing_input(const dyn_objective_in& in, int terms) {
#define NEED(bit, field) \
  if ((terms & (bit)) && in.field == nullptr) return #field
  const int charb_terms = DYN_OBJ_RGB | DYN_OBJ_TEMPORAL | DYN_OBJ_DYREGION | DYN_OBJ_DYNAMIC | DYN_OBJ_STATIC |
                          DYN_OBJ_BOOTSTRAP;
  NEED(charb_terms, gt_rgb);
  NEED(DYN_OBJ_RGB | DYN_OBJ_DYREGION | DYN_OBJ_DISP | DYN_OBJ_FLOW | DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA |
           DYN_OBJ_BOOTSTRAP, mask);
  NEED(DYN_OBJ_RGB, rgb);
  NEED(DYN_OBJ_TEMPORAL, a_rgb);
  NEED(DYN_OBJ_TEMPORAL, a_mask);
  NEED(DYN_OBJ_TEMPORAL, a_occ_map);
  NEED(DYN_OBJ_DYREGION | DYN_OBJ_DYNAMIC, motion_mask);
  NEED(DYN_OBJ_DYREGION, rgb_dy);
  NEED(DYN_OBJ_DYNAMIC, ref_dy_rgb);
  NEED(DYN_OBJ_DYNAMIC, ref_dy_mask);
  NEED(DYN_OBJ_DYNAMIC, a_dy_rgb);
  NEED(DYN_OBJ_DYNAMIC, a_dy_mask);
  NEED(DYN_OBJ_DYNAMIC, a_dy_occ_map);
  NEED(DYN_OBJ_DISP, depth);
  NEED(DYN_OBJ_DISP, disp);
  NEED(DYN_OBJ_FLOW, render_flows);
  NEED(DYN_OBJ_FLOW, flows);
  NEED(DYN_OBJ_FLOW, flow_masks);
  NEED(DYN_OBJ_CYCLE, pts_traj_ref);
  NEED(DYN_OBJ_CYCLE, pts_traj_anchor);
  NEED(DYN_OBJ_CYCLE, occ_weights);
  NEED(DYN_OBJ_REG, sf_seq);
  NEED(DYN_OBJ_ENTROPY | DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA, weights_dy);
  NEED(DYN_OBJ_ENTROPY | DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA, weights_st);
  NEED(DYN_OBJ_STATIC | DYN_OBJ_STATIC_EXTRA | DYN_OBJ_BOOTSTRAP, static_mask);
  NEED(DYN_OBJ_STATIC, rgb_static);
  NEED(DYN_OBJ_BOOTSTRAP, st_rgb);
  NEED(DYN_OBJ_DISTORTION, weights);
  if ((terms & DYN_OBJ_DISTORTION) && (in.dist_mid == nullptr) != (in.dist_interval == nullptr))
    return "dist_mid / dist_interval (both or neither)";
  if ((terms & DYN_OBJ_DISTORTION) && in.dist_mid == nullptr && in.s_vals == nullptr) return "s_vals";
#undef NEED
  return nullptr;
}

int check_in(const dyn_objective_in* in, int terms) {
  if (in == nullptr) return fail(DYN_E_INVALID, "dyn_objective: `in` is NULL");
  if (terms <= 0 || terms >= 2 * DYN_OBJ_BOOTSTRAP) return fail(DYN_E_INVALID, "dyn_objective: bad terms 0x%x", terms);
  if (in->R < 1) return fail(DYN_E_INVALID, "dyn_objective: R = %d (need >= 1)", in->R);
  const bool per_sample = terms & (DYN_OBJ_CYCLE | DYN_OBJ_REG | DYN_OBJ_ENTROPY | DYN_OBJ_STATIC |
                                   DYN_OBJ_STATIC_EXTRA | DYN_OBJ_DISTORTION);
  const int s_min = (terms & (DYN_OBJ_REG | DYN_OBJ_DISTORTION)) && !in->dist_mid ? 2 : 1;
  if (per_sample && in->S < s_min) return fail(DYN_E_INVALID, "dyn_objective: S = %d (need >= %d)", in->S, s_min);
  if ((terms & DYN_OBJ_CYCLE) && in->K < 1) return fail(DYN_E_INVALID, "dyn_objective: K = %d (need >= 1)", in->K);
  if ((terms & DYN_OBJ_REG) && in->T < 2) return fail(DYN_E_INVALID, "dyn_objective: T = %d (need >= 2)", in->T);
  if ((terms & DYN_OBJ_FLOW) && in->F < 1) return fail(DYN_E_INVALID, "dyn_objective: F = %d (need >= 1)", in->F);
  if (const char* m = missing_input(*in, terms))
    return fail(DYN_E_INVALID, "dyn_objective: an enabled term needs `%s` (NULL)", m);
  return DYN_OK;
}

size_t partial_bytes(int R) { return (size_t)cdiv(R < 1 ? 1 : R, kWarps) * S_NUM * sizeof(double); }

}  // namespace

}  // namespace dyn

using namespace dyn;

extern "C" {

size_t dyn_objective_workspace_bytes(int R) { return 256 + partial_bytes(R); }

int dyn_objective_sums(const dyn_objective_in* in, int terms, double* sums, void* workspace, size_t workspace_bytes,
                       void* stream) {
  if (int rc = check_in(in, terms)) return rc;
  DYN_CHECK_ARG(sums != nullptr && workspace != nullptr);
  if (workspace_bytes < dyn_objective_workspace_bytes(in->R))
    return fail(DYN_E_WORKSPACE, "dyn_objective_sums: workspace %zu < %zu bytes", workspace_bytes,
                dyn_objective_workspace_bytes(in->R));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(workspace);
  double* part = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 256);
  DYN_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), st));
  objective_sums_kernel<<<cdiv(in->R, kWarps), kWarps * 32, 0, st>>>(*in, terms, part, ticket, sums);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

int dyn_objective_finalize(const double* sums, int terms, const double* coef_host, float* loss, float* term_values,
                           double* scales, void* stream) {
  DYN_CHECK_ARG(sums && coef_host && loss && term_values && scales);
  DYN_CHECK_ARG(terms > 0 && terms < 2 * DYN_OBJ_BOOTSTRAP);
  Coef k;
  for (int i = 0; i < DYN_OBJ_NCOEF; ++i) k.c[i] = coef_host[i];
  objective_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(sums, terms, k, loss, term_values, scales);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

int dyn_objective_backward(const dyn_objective_in* in, int terms, const double* scales, const float* g_loss,
                           const float* g_terms, const dyn_objective_grad* grad, void* stream) {
  if (int rc = check_in(in, terms)) return rc;
  DYN_CHECK_ARG(scales != nullptr && grad != nullptr);
  objective_backward_kernel<<<cdiv(in->R, kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(*in, terms, scales, g_loss,
                                                                                        g_terms, *grad);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // extern "C"
