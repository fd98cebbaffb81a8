// Staged evaluation of the three networks (a3, a8-a11): the reference's op
// graph as one kernel per layer -- generic linear layers (fp32 SIMT in
// linear_f32.cu for DYN_PREC_FP32, tcgen05 in linear_tc.cu for DYN_PREC_BF16)
// plus the fused fp32 glue below (positional encodings, view
// pooling, visibility gating, ray transformer, heads).  This is the parity
// mode; the throughput mode is the tcgen05 path in nets_tc.cu.
#include <math.h>

#include "linear_tc.cuh"
#include "nets.cuh"
#include "nets_f32_bufs.cuh"
#include "nets_fused.cuh"
#include "fused_engine.cuh"

extern "C" long long* view_dbg_ptr();

namespace dyn {

// ---------------------------------------------------------------------------
// layouts
// ---------------------------------------------------------------------------
static LayerList* g_list = nullptr;  // layout being built (host, single-threaded at create time)

static LinearP take(int& off, int out, int in, bool bias = true) {
  LinearP l;
  l.in = in; l.out = out;
  l.w = off; off += out * in;
  if (bias) { l.b = off; off += out; } else { l.b = -1; }
  l.tc = g_list->packed_bytes;
  g_list->packed_bytes += (long long)((tc_packed_bytes(out, in) + 255) & ~(size_t)255);
  g_list->l[g_list->n++] = l;
  return l;
}

DynamicLayout dynamic_layout() {
  DynamicLayout L;
  int o = 0;
  L.all.n = 0; L.all.packed_bytes = 0;
  g_list = &L.all;
  L.ray_dir0 = take(o, 256, 21); L.ray_dir2 = take(o, kF, 256);
  L.base0 = take(o, 256, 3 * kF); L.base2 = take(o, 128, 256);
  L.vis0 = take(o, 128, 128); L.vis2 = take(o, 129, 128);
  L.vis2_0 = take(o, 128, 128); L.vis2_2 = take(o, 1, 128);
  L.geo0 = take(o, 256, 257); L.geo2 = take(o, 128, 256);
  L.wq = take(o, 128, 128, false); L.wk = take(o, 128, 128, false);
  L.wv = take(o, 128, 128, false); L.fc = take(o, 128, 128, false);
  L.ln_w = o; o += 128; L.ln_b = o; o += 128;
  L.refpts0 = take(o, 256, 161); L.refpts2 = take(o, 128, 256);
  L.outgeo0 = take(o, 128, 128); L.outgeo2 = take(o, 1, 128);
  L.rgb0 = take(o, 128, 155); L.rgb2 = take(o, 64, 128); L.rgb4 = take(o, 3, 64);
  L.total = o;
  return L;
}

StaticLayout static_layout(bool anti_alias) {
  StaticLayout L;
  int o = 0;
  L.all.n = 0; L.all.packed_bytes = 0;
  g_list = &L.all;
  L.s = -1;
  if (anti_alias) { L.s = o; o += 1; }
  L.ray_dir0 = take(o, 256, 103); L.ray_dir2 = take(o, kF, 256);
  L.ref_feat = take(o, kF, 66);
  L.base0 = take(o, 256, 6 * kF); L.base2 = take(o, 128, 256);
  L.vis0 = take(o, 128, 128); L.vis2 = take(o, 129, 128);
  L.vis2_0 = take(o, 128, 128); L.vis2_2 = take(o, 1, 128);
  L.geo0 = take(o, 256, 257); L.geo2 = take(o, 128, 256);
  L.wq = take(o, 128, 128, false); L.wk = take(o, 128, 128, false);
  L.wv = take(o, 128, 128, false); L.fc = take(o, 128, 128, false);
  L.ln_w = o; o += 128; L.ln_b = o; o += 128;
  L.outgeo0 = take(o, 128, 128); L.outgeo2 = take(o, 1, 128);
  L.rgb0 = take(o, 128, 261); L.rgb2 = take(o, 64, 128); L.rgb4 = take(o, 1, 64);
  L.total = o;
  return L;
}

MotionLayout motion_layout(int nb) {
  MotionLayout L;
  int o = 0;
  L.all.n = 0; L.all.packed_bytes = 0;
  g_list = &L.all;
  L.pts[0] = take(o, 256, 132);
  for (int i = 1; i < 8; ++i) L.pts[i] = take(o, 256, i == 5 ? 388 : 256);
  L.coeff = take(o, 3 * nb, 256);
  L.total = o;
  return L;
}

// ---------------------------------------------------------------------------
// a8 PeriodicEmbed (mlp_network.py:530-555): out = [x, cos(f_k x).., sin(f_k x)..]
// ---------------------------------------------------------------------------
struct PEFreqs {
  float f[16];
  int n;
};

PEFreqs pe_freqs(int n, bool linspace) {
  PEFreqs q;
  q.n = n;
  if (!linspace) {
    for (int k = 0; k < n; ++k) q.f[k] = (float)(1 << k);  // 2^k, mlp_network.py:546-547
  } else {
    // torch.linspace(1, n+1, n) (mlp_network.py:544): ATen fills the first half
    // from `start` and the second half from `end`.
    float start = 1.f, end = (float)(n + 1);
    float step = (end - start) / (float)(n - 1);
    int half = n / 2;
    for (int k = 0; k < n; ++k)
      q.f[k] = k < half ? start + step * (float)k : end - step * (float)(n - 1 - k);
  }
  return q;
}

// in [N, D] (ld = ldin), optional constant extra column appended (`extra`,
// used for the time channel of xyzt); out [N, Dt*(2n+1)] with Dt = D + has_extra
__global__ void pe_kernel(const float* __restrict__ in, int D, int ldin, int has_extra, float extra,
                          PEFreqs q, long long N, float* __restrict__ out) {
  const int Dt = D + has_extra;
  const int width = Dt * (2 * q.n + 1);
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * width) return;
  long long row = idx / width;
  int c = (int)(idx % width);
  int blk = c / Dt, d = c % Dt;
  float x = d < D ? in[row * ldin + d] : extra;
  float v;
  if (blk == 0) v = x;
  else if (blk <= q.n) v = cosf(q.f[blk - 1] * x);
  else v = sinf(q.f[blk - 1 - q.n] * x);
  out[idx] = v;
}

static int launch_pe(const float* in, int D, int ldin, int has_extra, float extra, int n,
                     bool linspace, long long N, float* out, cudaStream_t st) {
  if (N == 0) return DYN_OK;
  int width = (D + has_extra) * (2 * n + 1);
  pe_kernel<<<cdiv(N * width, 256), 256, 0, st>>>(in, D, ldin, has_extra, extra, pe_freqs(n, linspace),
                                                  N, out);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

// ---------------------------------------------------------------------------
// view pooling, stage 1
// ---------------------------------------------------------------------------
// dynamic: feat = rgb_feat + dfeat; weight = mask/(sum mask + 1e-8); mean/var
// (mlp_network.py:244-262).  Thread per (point, channel).
__global__ void dyn_pool1_kernel(const float* __restrict__ rgb_feat, const float* __restrict__ dfeat,
                                 const float* __restrict__ mask, long long P, int V,
                                 float* __restrict__ feat, float* __restrict__ mv /* [P,70] */,
                                 float* __restrict__ weight) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * kF) return;
  long long p = idx / kF;
  int c = (int)(idx % kF);
  float msum = 0.f;
  for (int v = 0; v < V; ++v) msum += mask[p * V + v];
  float den = msum + 1e-8f;
  float d = dfeat[c];
  float mean = 0.f;
  for (int v = 0; v < V; ++v) {
    float f = rgb_feat[(p * V + v) * kF + c] + d;
    feat[(p * V + v) * kF + c] = f;
    float w = mask[p * V + v] / den;
    if (c == 0) weight[p * V + v] = w;
    mean += f * w;
  }
  float var = 0.f;
  for (int v = 0; v < V; ++v) {
    float f = rgb_feat[(p * V + v) * kF + c] + d;
    float w = mask[p * V + v] / den;
    float t = f - mean;
    var += w * t * t;
  }
  mv[p * 2 * kF + c] = mean;
  mv[p * 2 * kF + kF + c] = var;
}

// static: feat70 = [rgb_feat, src_feat * ref_feat]; optional mask_rgb gating;
// anti-alias or plain pooling weights; mean/var (mlp_network.py:452-477).
__global__ void st_pool1_kernel(const float* __restrict__ rgb_feat, const float* __restrict__ src_feat,
                                const float* __restrict__ ref_feat, const float* __restrict__ ray_diff,
                                const float* __restrict__ mask_in, const float* __restrict__ s_param,
                                int mask_rgb, long long P, int S, int V, float* __restrict__ feat70,
                                float* __restrict__ mv /* [P,140] */, float* __restrict__ weight,
                                float* __restrict__ mask_eff) {
  const int F2 = 2 * kF;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * F2) return;
  long long p = idx / F2;
  int c = (int)(idx % F2);
  long long ray = p / S;
  float w[kMaxViews];
  float emin = INFINITY, wsum = 0.f;
  float sabs = s_param ? fabsf(*s_param) : 0.f;
  for (int v = 0; v < V; ++v) {
    long long m = p * V + v;
    float mk = mask_in[m];
    if (mask_rgb) {
      const float* rf = rgb_feat + m * kF;
      mk *= ((rf[0] + rf[1] + rf[2]) > 1e-3f) ? 1.f : 0.f;
    }
    if (c == 0) mask_eff[m] = mk;
    if (s_param) {
      float e = expf(sabs * (ray_diff[m * 4 + 3] - 1.f));
      emin = fminf(emin, e);
      w[v] = e;
    } else {
      w[v] = mk;
      wsum += mk;
    }
  }
  if (s_param) {
    for (int v = 0; v < V; ++v) {
      long long m = p * V + v;
      float mk = mask_in[m];
      if (mask_rgb) {
        const float* rf = rgb_feat + m * kF;
        mk *= ((rf[0] + rf[1] + rf[2]) > 1e-3f) ? 1.f : 0.f;
      }
      w[v] = (w[v] - emin) * mk;
      wsum += w[v];
    }
  }
  float den = wsum + 1e-8f;
  float mean = 0.f;
  float fv[kMaxViews];
  for (int v = 0; v < V; ++v) {
    long long m = p * V + v;
    float f = c < kF ? rgb_feat[m * kF + c] : src_feat[m * kF + (c - kF)] * ref_feat[ray * kF + (c - kF)];
    fv[v] = f;
    feat70[m * F2 + c] = f;
    float wn = w[v] / den;
    w[v] = wn;
    if (c == 0) weight[m] = wn;
    mean += f * wn;
  }
  float var = 0.f;
  for (int v = 0; v < V; ++v) {
    float t = fv[v] - mean;
    var += w[v] * t * t;
  }
  mv[p * 2 * F2 + c] = mean;
  mv[p * 2 * F2 + F2 + c] = var;
}

// x += x_res ; vis = sigmoid(x_vis[128]) * mask   (mlp_network.py:273-275)
// (x2 may alias x: inference updates x in place, training keeps both)
__global__ void vis1_kernel(const float* x, const float* __restrict__ xvis,
                            const float* __restrict__ mask, long long M, float* x2, float* __restrict__ vis) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * 128) return;
  long long m = idx >> 7;
  int c = (int)(idx & 127);
  x2[idx] = x[idx] + xvis[m * 129 + c];
  if (c == 0) vis[m] = sigmoid_f(xvis[m * 129 + 128]) * mask[m];
}

// vis2 = vis2raw*mask; weight = vis2/(sum+1e-8); weighted mean/var of x over
// views; G = [mean128, var128, mean_v(weight)]; nvalid = sum mask
// (mlp_network.py:276-284).  Thread per (point, channel).
__global__ void pool2_kernel(const float* __restrict__ x, float* __restrict__ vis2,
                             const float* __restrict__ mask, long long P, int V,
                             float* __restrict__ G /* [P,257] */, float* __restrict__ nvalid) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * 128) return;
  long long p = idx >> 7;
  int c = (int)(idx & 127);
  float w[kMaxViews];
  float sum = 0.f, ms = 0.f;
  for (int v = 0; v < V; ++v) {
    float mk = mask[p * V + v];
    float t = vis2[p * V + v] * mk;
    w[v] = t;
    sum += t;
    ms += mk;
  }
  float den = sum + 1e-8f;
  float mean = 0.f, wmean = 0.f;
  for (int v = 0; v < V; ++v) {
    w[v] = w[v] / den;
    wmean += w[v];
    mean += x[(p * V + v) * 128 + c] * w[v];
  }
  float var = 0.f;
  for (int v = 0; v < V; ++v) {
    float t = x[(p * V + v) * 128 + c] - mean;
    var += w[v] * t * t;
  }
  G[p * 257 + c] = mean;
  G[p * 257 + 128 + c] = var;
  __syncwarp();
  if (c == 0) {
    G[p * 257 + 256] = wmean / (float)V;  // weight.mean(dim=2)
    nvalid[p] = ms;
  }
}

// second pass writes the masked visibility back (needed by the static RGB
// head, mlp_network.py:489,513); separate kernel to avoid a read/write race
// with pool2's readers.
__global__ void mask_vis2_kernel(float* __restrict__ vis2, const float* __restrict__ mask, long long M) {
  long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m < M) vis2[m] *= mask[m];
}

// g[p, :] += sinusoid[s, :]  (mlp_network.py:220-234, :286); table built on
// the fly in double precision like the reference's numpy code.
__global__ void add_posenc_kernel(float* __restrict__ g, long long P, int S) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * 128) return;
  int s = (int)((idx >> 7) % S);
  int j = (int)(idx & 127);
  double ang = (double)s / pow(10000.0, 2.0 * (double)(j / 2) / 128.0);
  g[idx] += (float)((j & 1) ? cos(ang) : sin(ang));
}

// sinusoid table [S,128] (mlp_network.py:220-234), double precision like numpy
__global__ void posenc_table_kernel(float* __restrict__ tab, int S) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * 128) return;
  int s = idx >> 7, j = idx & 127;
  double ang = (double)s / pow(10000.0, 2.0 * (double)(j / 2) / 128.0);
  tab[idx] = (float)((j & 1) ? cos(ang) : sin(ang));
}

// ---------------------------------------------------------------------------
// a11 ray transformer core: softmax(q k^T / sqrt(dk)) v per ray and head.
// Block per ray, thread per query sample, K/V of one head staged in smem.
// Masked QUERY rows get all logits = -1e9 -> uniform attention
// (mlp_network.py:23-24, :91-94).
// ---------------------------------------------------------------------------
// 4 consecutive elements of a [*,128] row stored as fp32 or bf16
// BF: `base` is a bf16 tile image with 16 k-groups (fused_engine.cuh), elem = row * 128 + col
template <bool BF>
__device__ __forceinline__ float4 ld4(const void* base, long long elem) {
  if (BF) {
    const long long row = elem >> 7;
    const int col = (int)(elem & 127);
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(base) +
                                                    fe::tile_image_off(row, col >> 3, 16) + (col & 7) * 2);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
    return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + elem);
}
template <bool BF>
__device__ __forceinline__ void st4(void* base, long long elem, float4 v) {
  if (BF) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&a); u.y = *reinterpret_cast<uint32_t*>(&b);
    const long long row = elem >> 7;
    const int col = (int)(elem & 127);
    *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(base) + fe::tile_image_off(row, col >> 3, 16) +
                              (col & 7) * 2) = u;
  } else {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + elem) = v;
  }
}

// BF: Q/K/V/O are bf16 tile images (fused path) instead of fp32 rows (staged path)
template <bool BF>
__global__ void attention_kernel(const void* __restrict__ Q, const void* __restrict__ K,
                                 const void* __restrict__ Vv, const float* __restrict__ nvalid, int S,
                                 void* __restrict__ O) {
  extern __shared__ __align__(16) float sm[];
  float4* Ks = reinterpret_cast<float4*>(sm);          // [S][8] float4 = 32 floats per key
  float4* Vs = reinterpret_cast<float4*>(sm) + S * 8;  // [S][8]
  const int ray = blockIdx.x;
  const int i = threadIdx.x;
  const long long base = (long long)ray * S;
  const bool row_ok = (i < S) && (nvalid[base + i] > 1.f);
  const float inv_temp = 1.f / sqrtf(32.f);
  for (int h = 0; h < 4; ++h) {
    __syncthreads();
    for (int e = threadIdx.x; e < S * 8; e += blockDim.x) {
      int j = e >> 3, d4 = e & 7;
      Ks[e] = ld4<BF>(K, (base + j) * 128 + h * 32 + d4 * 4);
      Vs[e] = ld4<BF>(Vv, (base + j) * 128 + h * 32 + d4 * 4);
    }
    __syncthreads();
    if (i < S) {
      float q[32], o[32];
#pragma unroll
      for (int d4 = 0; d4 < 8; ++d4) {
        float4 t = ld4<BF>(Q, (base + i) * 128 + h * 32 + d4 * 4);
        q[4 * d4] = t.x * inv_temp; q[4 * d4 + 1] = t.y * inv_temp;
        q[4 * d4 + 2] = t.z * inv_temp; q[4 * d4 + 3] = t.w * inv_temp;
      }
#pragma unroll
      for (int d = 0; d < 32; ++d) o[d] = 0.f;
      float mx = -INFINITY, den = 0.f;
      for (int j = 0; j < S; ++j) {
        float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
#pragma unroll
        for (int d4 = 0; d4 < 8; ++d4) {
          const float4 kk = Ks[j * 8 + d4];  // same address in every lane: broadcast
          l0 = fmaf(q[4 * d4], kk.x, l0); l1 = fmaf(q[4 * d4 + 1], kk.y, l1);
          l2 = fmaf(q[4 * d4 + 2], kk.z, l2); l3 = fmaf(q[4 * d4 + 3], kk.w, l3);
        }
        float l = (l0 + l1) + (l2 + l3);
        if (!row_ok) l = -1e9f;
        const float mn = fmaxf(mx, l);
        const float corr = __expf(mx - mn);
        const float pj = __expf(l - mn);
        den = den * corr + pj;
        if (mn != mx) {  // rescale only when the running max moved
#pragma unroll
          for (int d = 0; d < 32; ++d) o[d] *= corr;
        }
#pragma unroll
        for (int d4 = 0; d4 < 8; ++d4) {
          const float4 vv = Vs[j * 8 + d4];
          o[4 * d4] = fmaf(pj, vv.x, o[4 * d4]); o[4 * d4 + 1] = fmaf(pj, vv.y, o[4 * d4 + 1]);
          o[4 * d4 + 2] = fmaf(pj, vv.z, o[4 * d4 + 2]); o[4 * d4 + 3] = fmaf(pj, vv.w, o[4 * d4 + 3]);
        }
        mx = mn;
      }
      const float inv = 1.f / den;
#pragma unroll
      for (int d4 = 0; d4 < 8; ++d4)
        st4<BF>(O, (base + i) * 128 + h * 32 + d4 * 4,
                make_float4(o[4 * d4] * inv, o[4 * d4 + 1] * inv, o[4 * d4 + 2] * inv, o[4 * d4 + 3] * inv));
    }
  }
}

// out = LayerNorm(a + resid) * w + b, eps 1e-6 (mlp_network.py:100-102). Warp per row.
__global__ void resid_ln_kernel(const float* __restrict__ a, const float* __restrict__ resid,
                                const float* __restrict__ w, const float* __restrict__ b, long long P,
                                float* __restrict__ out) {
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= P) return;
  float v[4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int c = lane + 32 * i;
    v[i] = a[row * 128 + c] + resid[row * 128 + c];
    s += v[i];
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  float mean = s / 128.f;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) { float t = v[i] - mean; q += t * t; }
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  float rstd = rsqrtf(q / 128.f + 1e-6f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int c = lane + 32 * i;
    out[row * 128 + c] = (v[i] - mean) * rstd * w[c] + b[c];
  }
}

// dynamic head output: raw = [rgb (0 where no valid view), sigma - shift (-1e9 where no valid view)]
// (mlp_network.py:294-315)
__global__ void dyn_out_kernel(const float* __restrict__ rgb, const float* __restrict__ sigma,
                               const float* __restrict__ nvalid, float shift, long long P,
                               float* __restrict__ raw) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  bool none = nvalid[p] < 1.f;
  float4 o;
  o.x = none ? 0.f : rgb[p * 3];
  o.y = none ? 0.f : rgb[p * 3 + 1];
  o.z = none ? 0.f : rgb[p * 3 + 2];
  o.w = none ? -1e9f : sigma[p] - shift;
  reinterpret_cast<float4*>(raw)[p] = o;
}

// static head output: masked softmax over views of the blending logits, blend
// the gathered source colours (mlp_network.py:503-526)
__global__ void st_out_kernel(const float* __restrict__ logit, const float* __restrict__ mask_eff,
                              const float* __restrict__ rgb_feat, const float* __restrict__ sigma,
                              const float* __restrict__ nvalid, long long P, int V, int ldf,
                              float* __restrict__ raw) {
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float l[kMaxViews];
  float mx = -INFINITY;
  for (int v = 0; v < V; ++v) {
    float t = mask_eff[p * V + v] == 0.f ? -1e9f : logit[p * V + v];
    l[v] = t;
    mx = fmaxf(mx, t);
  }
  float den = 0.f;
  for (int v = 0; v < V; ++v) { l[v] = expf(l[v] - mx); den += l[v]; }
  float r = 0.f, g = 0.f, b = 0.f;
  for (int v = 0; v < V; ++v) {
    float w = l[v] / den;
    const float* c = rgb_feat + (p * V + v) * ldf;
    r += c[0] * w; g += c[1] * w; b += c[2] * w;
  }
  float4 o = make_float4(r, g, b, nvalid[p] < 1.f ? -1e9f : sigma[p]);
  reinterpret_cast<float4*>(raw)[p] = o;
}

// time feature of the dynamic net: ray_dir_fc(PE(t)) -> 35 values, identical
// for every (ray, sample, view) of a call (mlp_network.py:240-244). One block.
// `keep` (training): dfeat[64..319] = hidden activations, dfeat[320..340] = PE(t)
__global__ void dyn_time_feat_kernel(const float* __restrict__ prm, DynamicLayout L, float t,
                                     float* __restrict__ dfeat, int keep) {
  __shared__ float pe[21];
  __shared__ float h[256];
  int tid = threadIdx.x;
  if (tid < 21) {
    float v;
    if (tid == 0) v = t;
    else if (tid <= 10) v = cosf((float)(1 << (tid - 1)) * t);
    else v = sinf((float)(1 << (tid - 11)) * t);
    pe[tid] = v;
  }
  __syncthreads();
  {
    float s = prm[L.ray_dir0.b + tid];
    for (int k = 0; k < 21; ++k) s = fmaf(prm[L.ray_dir0.w + tid * 21 + k], pe[k], s);
    h[tid] = elu_f(s);
    if (keep) {
      dfeat[64 + tid] = h[tid];
      if (tid < 21) dfeat[320 + tid] = pe[tid];
    }
  }
  __syncthreads();
  if (tid < kF) {
    float s = prm[L.ray_dir2.b + tid];
    for (int k = 0; k < 256; ++k) s = fmaf(prm[L.ray_dir2.w + tid * 256 + k], h[k], s);
    dfeat[tid] = elu_f(s);
  }
}

__global__ void zero_last_kernel(float* __restrict__ coeff, int R, int S, int n_last, int width) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long tot = (long long)R * n_last * width;
  if (idx >= tot) return;
  int c = (int)(idx % width);
  long long t = idx / width;
  int s = S - n_last + (int)(t % n_last);
  long long r = t / n_last;
  coeff[(r * S + s) * width + c] *= 0.0f;  // reference multiplies by 0 (render_ray.py:472)
}

static const float* P_(const dyn_net* n, int off) { return off < 0 ? nullptr : n->params + off; }

// one linear layer in the requested precision: tcgen05 (bf16 operands) when the
// net carries packed images and the layer is big enough to fill a UMMA tile
static int run_lin(const dyn_net* n, const LinearP& l, const LinArgs& a, int prec, cudaStream_t st) {
  if (prec == DYN_PREC_BF16 && n->packed != nullptr && a.M >= 128 && l.out >= 16)
    return launch_linear_tc(a, reinterpret_cast<const char*>(n->packed) + l.tc, st);
  return launch_linear(a, st);
}
static LinArgs L1(const dyn_net* n, const LinearP& l, const float* X, float* Y, long long M, int act) {
  return lin1(X, l.in, P_(n, l.w), P_(n, l.b), Y, l.out, M, l.out, l.in, act);
}

#define RUN(expr)            \
  do {                       \
    int rc_ = (expr);        \
    if (rc_) return rc_;     \
  } while (0)

int net_rows_per_chunk(int S, int V) {
  long long rows = 4194304;  // (point, view) rows per internal chunk (workspace ~1.5 KB/row)
  long long r = rows / ((long long)S * V);
  return (int)(r < 1 ? 1 : r);
}

// per-point tail shared by the staged and the fused paths:
// geometry_fc -> (+ sinusoid) -> ray transformer -> t.G3   (mlp_network.py:283-289 / :496-502)
template <class Layout>
static int run_point_tail(const dyn_net* n, const Layout& L, const float* G, int ldg, long long P,
                          int R, int S, bool add_posenc, TrunkBufs& t, int prec, cudaStream_t st) {
  // geometry_fc (:283 / :496)
  {
    LinArgs ga = L1(n, L.geo0, G, t.GH, P, ACT_ELU);
    ga.seg[0].ld = ldg;
    RUN(run_lin(n, L.geo0, ga, prec, st));
  }
  RUN(run_lin(n, L.geo2, L1(n, L.geo2, t.GH, t.G2, P, ACT_ELU), prec, st));
  if (add_posenc) {
    add_posenc_kernel<<<cdiv(P * 128, 256), 256, 0, st>>>(t.G2, P, S);
    DYN_LAUNCH_CHECK();
  }
  // ray transformer (:287 / :500)
  RUN(run_lin(n, L.wq, L1(n, L.wq, t.G2, t.Q, P, ACT_NONE), prec, st));
  RUN(run_lin(n, L.wk, L1(n, L.wk, t.G2, t.K, P, ACT_NONE), prec, st));
  RUN(run_lin(n, L.wv, L1(n, L.wv, t.G2, t.V, P, ACT_NONE), prec, st));
  {
    int threads = ((S + 31) / 32) * 32;
    size_t smem = (size_t)2 * S * 32 * sizeof(float);
    if (threads > 1024) return fail(DYN_E_INVALID, "ray transformer supports S <= 1024 (got %d)", S);
    if (smem > 48 * 1024)
      DYN_CUDA(cudaFuncSetAttribute(attention_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    attention_kernel<false><<<R, threads, smem, st>>>(t.Q, t.K, t.V, t.nvalid, S, t.O);
    DYN_LAUNCH_CHECK();
  }
  RUN(run_lin(n, L.fc, L1(n, L.fc, t.O, t.O2, P, ACT_NONE), prec, st));
  resid_ln_kernel<<<cdiv(P * 32, 256), 256, 0, st>>>(t.O2, t.G2, P_(n, L.ln_w), P_(n, L.ln_b), P, t.G3);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

template <class Layout>
static int run_trunk(const dyn_net* n, const Layout& L, const Seg& mv, const Seg& feat,
                     const float* weight1, const float* mask, long long M, long long P, int R,
                     int S, int V, bool add_posenc, TrunkBufs& t, int prec, cudaStream_t st) {
  // base_fc (mlp_network.py:270 / :483)
  LinArgs a = L1(n, L.base0, nullptr, t.H1, M, ACT_ELU);
  a.seg[0] = mv; a.seg[1] = feat; a.nseg = 2;
  RUN(run_lin(n, L.base0, a, prec, st));
  RUN(run_lin(n, L.base2, L1(n, L.base2, t.H1, t.X, M, ACT_ELU), prec, st));
  // vis_fc(x * weight) (:272 / :485)
  a = L1(n, L.vis0, t.X, t.H2, M, ACT_ELU);
  a.row_scale = weight1;
  RUN(run_lin(n, L.vis0, a, prec, st));
  RUN(run_lin(n, L.vis2, L1(n, L.vis2, t.H2, t.XV, M, ACT_ELU), prec, st));
  vis1_kernel<<<cdiv(M * 128, 256), 256, 0, st>>>(t.X, t.XV, mask, M, t.X2, t.vis1);
  DYN_LAUNCH_CHECK();
  // vis_fc2(x * vis) (:276 / :489)
  a = L1(n, L.vis2_0, t.X2, t.H3, M, ACT_ELU);
  a.row_scale = t.vis1;
  RUN(run_lin(n, L.vis2_0, a, prec, st));
  RUN(run_lin(n, L.vis2_2, L1(n, L.vis2_2, t.H3, t.vis2, M, ACT_SIGMOID), prec, st));
  pool2_kernel<<<cdiv(P * 128, 256), 256, 0, st>>>(t.X2, t.vis2, mask, P, V, t.G, t.nvalid);
  DYN_LAUNCH_CHECK();
  mask_vis2_kernel<<<cdiv(M, 256), 256, 0, st>>>(t.vis2, mask, M);
  DYN_LAUNCH_CHECK();
  return run_point_tail(n, L, t.G, 257, P, R, S, add_posenc, t, prec, st);
}

// ---------------------------------------------------------------------------
// DynibarDynamic.forward, fp32 (mlp_network.py:236-316)
// ---------------------------------------------------------------------------
size_t net_dynamic_f32_workspace(int R, int S, int V) {
  Bump b{nullptr, 0};
  DynBufs d;
  int rc = net_rows_per_chunk(S, V);
  return dyn_alloc(b, R < rc ? R : rc, S, V, &d);
}

int net_dynamic_f32(const dyn_net* n, const float* pts, const float* rgb_feat, const float* ray_dir,
                    const float* mask, float time, int R_all, int S, int V, float* raw, void* ws,
                    size_t ws_bytes, int prec, cudaStream_t st, bool train) {
  const DynamicLayout& L = n->dl;
  const int RC = net_rows_per_chunk(S, V);
  if (train && R_all > RC) return fail(DYN_E_INVALID, "training forward: %d rays exceed one internal chunk (%d)", R_all, RC);
  for (int r0 = 0; r0 < R_all; r0 += RC) {
    const int R = (R_all - r0) < RC ? (R_all - r0) : RC;
    const long long P = (long long)R * S, M = P * V, p0 = (long long)r0 * S;
    Bump b{(char*)ws, 0};
    DynBufs d;
    if (dyn_alloc(b, R, S, V, &d, train) > ws_bytes)
      return fail(DYN_E_WORKSPACE, "net_dynamic: workspace %zu < %zu", ws_bytes, b.off);
    const float* c_pts = pts + p0 * 3;
    const float* c_feat = rgb_feat + p0 * V * kF;
    const float* c_mask = mask + p0 * V;
    dyn_time_feat_kernel<<<1, 256, 0, st>>>(n->params, L, time, d.dfeat, train ? 1 : 0);
    DYN_LAUNCH_CHECK();
    dyn_pool1_kernel<<<cdiv(P * kF, 256), 256, 0, st>>>(c_feat, d.dfeat, c_mask, P, V, d.feat, d.mv, d.w1);
    DYN_LAUNCH_CHECK();
    RUN(run_trunk(n, L, Seg{d.mv, 2 * kF, 2 * kF, V}, Seg{d.feat, kF, kF, 1}, d.w1, c_mask, M, P, R, S,
                  V, /*add_posenc=*/true, d.t, prec, st));
    // ref_pts_fc(cat[g, PE(pts)]) (:291-292)
    RUN(launch_pe(c_pts, 3, 3, 0, 0.f, 5, false, P, d.ptspe, st));
    LinArgs a = L1(n, L.refpts0, nullptr, d.G4h, P, ACT_ELU);
    a.seg[0] = Seg{d.t.G3, 128, 128, 1}; a.seg[1] = Seg{d.ptspe, 33, 33, 1}; a.nseg = 2;
    RUN(run_lin(n, L.refpts0, a, prec, st));
    RUN(run_lin(n, L.refpts2, L1(n, L.refpts2, d.G4h, d.G4, P, ACT_ELU), prec, st));
    // sigma head (:294-299)
    RUN(run_lin(n, L.outgeo0, L1(n, L.outgeo0, d.G4, d.sh, P, ACT_ELU), prec, st));
    RUN(run_lin(n, L.outgeo2, L1(n, L.outgeo2, d.sh, d.sig, P, ACT_NONE), prec, st));
    // rgb head (:301-314)
    RUN(launch_pe(ray_dir + (long long)r0 * 3, 3, 3, 0, 0.f, 4, false, R, d.dirpe, st));
    a = L1(n, L.rgb0, nullptr, d.ch, P, ACT_ELU);
    a.seg[0] = Seg{d.G4, 128, 128, 1}; a.seg[1] = Seg{d.dirpe, 27, 27, S}; a.nseg = 2;
    RUN(run_lin(n, L.rgb0, a, prec, st));
    RUN(run_lin(n, L.rgb2, L1(n, L.rgb2, d.ch, d.ch2, P, ACT_ELU), prec, st));
    RUN(run_lin(n, L.rgb4, L1(n, L.rgb4, d.ch2, d.rgb, P, ACT_SIGMOID), prec, st));
    dyn_out_kernel<<<cdiv(P, 256), 256, 0, st>>>(d.rgb, d.sig, d.t.nvalid, n->shift, P, raw + p0 * 4);
    DYN_LAUNCH_CHECK();
  }
  return DYN_OK;
}

// ---------------------------------------------------------------------------
// DynibarStatic.forward, fp32 (mlp_network.py:423-527)
// ---------------------------------------------------------------------------
size_t net_static_f32_workspace(int R, int S, int V) {
  Bump b{nullptr, 0};
  StBufs d;
  int rc = net_rows_per_chunk(S, V);
  return st_alloc(b, R < rc ? R : rc, S, V, &d);
}

int net_static_f32(const dyn_net* n, const float* pts, const float* ref_rays, const float* src_rays,
                   const float* rgb_feat, const float* ray_diff, const float* mask, int R_all, int S,
                   int V, float* raw, void* ws, size_t ws_bytes, int prec, cudaStream_t st, bool train) {
  const StaticLayout& L = n->sl;
  const int RC = net_rows_per_chunk(S, V);
  if (train && R_all > RC) return fail(DYN_E_INVALID, "training forward: %d rays exceed one internal chunk (%d)", R_all, RC);
  for (int r0 = 0; r0 < R_all; r0 += RC) {
    const int R = (R_all - r0) < RC ? (R_all - r0) : RC;
    const long long P = (long long)R * S, M = P * V, p0 = (long long)r0 * S;
    Bump b{(char*)ws, 0};
    StBufs d;
    if (st_alloc(b, R, S, V, &d, train) > ws_bytes)
      return fail(DYN_E_WORKSPACE, "net_static: workspace %zu < %zu", ws_bytes, b.off);
    const float* c_feat = rgb_feat + p0 * V * kF;
    const float* c_rd = ray_diff + p0 * V * 4;
    const float* c_mask = mask + p0 * V;
    // positional encodings (:434-436)
    RUN(launch_pe(pts + p0 * 3, 3, 3, 0, 0.f, 5, false, P, d.ptspe, st));
    RUN(launch_pe(src_rays + p0 * V * 6, 6, 6, 0, 0.f, 5, false, M, d.srcpe, st));
    RUN(launch_pe(ref_rays + (long long)r0 * 6, 6, 6, 0, 0.f, 5, false, R, d.refpe, st));
    // src_feat = ray_dir_fc([pts_pe, src_pe, ray_diff]) (:441-449)
    LinArgs a = L1(n, L.ray_dir0, nullptr, d.H0, M, ACT_ELU);
    a.seg[0] = Seg{d.ptspe, 33, 33, V}; a.seg[1] = Seg{d.srcpe, 66, 66, 1};
    a.seg[2] = Seg{c_rd, 4, 4, 1}; a.nseg = 3;
    RUN(run_lin(n, L.ray_dir0, a, prec, st));
    RUN(run_lin(n, L.ray_dir2, L1(n, L.ray_dir2, d.H0, d.SF, M, ACT_NONE), prec, st));
    // ref_feat = ref_feature_fc(ref_pe) per ray (:450)
    RUN(run_lin(n, L.ref_feat, L1(n, L.ref_feat, d.refpe, d.reff, R, ACT_NONE), prec, st));
    st_pool1_kernel<<<cdiv(P * 2 * kF, 256), 256, 0, st>>>(
        c_feat, d.SF, d.reff, c_rd, c_mask, n->anti_alias ? n->params + L.s : nullptr, n->mask_rgb, P,
        S, V, d.feat70, d.mv, d.w1, d.meff);
    DYN_LAUNCH_CHECK();
    RUN(run_trunk(n, L, Seg{d.mv, 4 * kF, 4 * kF, V}, Seg{d.feat70, 2 * kF, 2 * kF, 1}, d.w1, d.meff,
                  M, P, R, S, V, /*add_posenc=*/false, d.t, prec, st));
    // sigma head (:503-506)
    RUN(run_lin(n, L.outgeo0, L1(n, L.outgeo0, d.t.G3, d.sh, P, ACT_ELU), prec, st));
    RUN(run_lin(n, L.outgeo2, L1(n, L.outgeo2, d.sh, d.sig, P, ACT_NONE), prec, st));
    // rgb blending head on [g, x, vis, ray_diff] (:508-525)
    a = L1(n, L.rgb0, nullptr, d.ch, M, ACT_ELU);
    a.seg[0] = Seg{d.t.G3, 128, 128, V}; a.seg[1] = Seg{d.t.X2, 128, 128, 1};
    a.seg[2] = Seg{d.t.vis2, 1, 1, 1}; a.seg[3] = Seg{c_rd, 4, 4, 1}; a.nseg = 4;
    RUN(run_lin(n, L.rgb0, a, prec, st));
    RUN(run_lin(n, L.rgb2, L1(n, L.rgb2, d.ch, d.ch2, M, ACT_ELU), prec, st));
    RUN(run_lin(n, L.rgb4, L1(n, L.rgb4, d.ch2, d.logit, M, ACT_NONE), prec, st));
    st_out_kernel<<<cdiv(P, 256), 256, 0, st>>>(d.logit, d.meff, c_feat, d.sig, d.t.nvalid, P, V, kF,
                                                raw + p0 * 4);
    DYN_LAUNCH_CHECK();
  }
  return DYN_OK;
}

// ---------------------------------------------------------------------------
// MotionMLP.forward, fp32 (mlp_network.py:605-618)
// ---------------------------------------------------------------------------
static const long long kMotionRows = 262144;

size_t motion_f32_workspace(long long N) {
  long long n = N < kMotionRows ? N : kMotionRows;
  Bump b{nullptr, 0};
  b.f(n * 132); b.f(n * 256); b.f(n * 256);
  return b.off;
}

// xyz [N,3] + constant time, or xyzt [N,4] when time_is_column
int motion_f32(const dyn_net* n, const float* x, int ldx, bool time_is_column, float time,
               long long N_all, float* coeff, void* ws, size_t ws_bytes, int prec, cudaStream_t st) {
  const MotionLayout& L = n->ml;
  if (prec == DYN_PREC_BF16 && n->motion.img != nullptr) {
    // whole MLP in one tcgen05 kernel (chains_fused.cu); no workspace needed
    MotionFusedArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.ldx = ldx; a.time_is_column = time_is_column ? 1 : 0; a.time = time;
    a.N = N_all; a.S = 0; a.n_last = 0; a.coeff = coeff;
    return launch_motion_fused(n, a, st);
  }
  for (long long i0 = 0; i0 < N_all; i0 += kMotionRows) {
    long long N = (N_all - i0) < kMotionRows ? (N_all - i0) : kMotionRows;
    Bump b{(char*)ws, 0};
    float* X0 = b.f(N * 132);
    float* A = b.f(N * 256);
    float* B = b.f(N * 256);
    if (b.off > ws_bytes) return fail(DYN_E_WORKSPACE, "motion: workspace %zu < %zu", ws_bytes, b.off);
    if (time_is_column)
      RUN(launch_pe(x + i0 * ldx, 4, ldx, 0, 0.f, 16, true, N, X0, st));
    else
      RUN(launch_pe(x + i0 * ldx, 3, ldx, 1, time, 16, true, N, X0, st));
    float *cur = A, *nxt = B;
    RUN(run_lin(n, L.pts[0], L1(n, L.pts[0], X0, cur, N, ACT_RELU), prec, st));
    for (int i = 1; i < 8; ++i) {
      LinArgs a = L1(n, L.pts[i], cur, nxt, N, ACT_RELU);
      if (i == 5) {  // skip connection: input is cat([input_pts, h]) (:612-613)
        a.seg[0] = Seg{X0, 132, 132, 1};
        a.seg[1] = Seg{cur, 256, 256, 1};
        a.nseg = 2;
      }
      RUN(run_lin(n, L.pts[i], a, prec, st));
      float* t = cur; cur = nxt; nxt = t;
    }
    RUN(run_lin(n, L.coeff, L1(n, L.coeff, cur, coeff + i0 * L.coeff.out, N, ACT_NONE), prec, st));
  }
  return DYN_OK;
}

// hooks for the training slice (motion_train.cu): the embedding of xyzt [N,4] and its frequencies
int motion_embed(const float* xyzt, long long N, float* x0, cudaStream_t st) {
  return launch_pe(xyzt, 4, 4, 0, 0.f, 16, true, N, x0, st);
}
void motion_freqs(float f[16]) {
  const PEFreqs q = pe_freqs(16, true);
  for (int k = 0; k < 16; ++k) f[k] = q.f[k];
}

// ---------------------------------------------------------------------------
// Fused (DYN_PREC_BF16) evaluation: per-view stage in ONE tcgen05 kernel
// (nets_fused.cu: projection + gather + per-view MLP chain + pooling), then the
// per-point tail and heads as staged tensor-core layers.
// ---------------------------------------------------------------------------
struct FusedBufs {
  float *small, *refpl, *refpe, *reff, *G, *X, *vis2, *rd, *meff, *rgbin;
  float *ptspe, *dirpe, *G4h, *G4, *sh, *sig, *ch, *ch2, *rgb, *logit;
  TrunkBufs t;
};

static size_t fused_alloc(Bump& b, bool st_net, int R, int S, int V, FusedBufs* d) {
  const long long P = (long long)R * S, M = P * V;
  d->small = b.f(64);
  d->G = b.f(((P + 255) / 256) * 256 * (kGStride / 2));  // bf16 tile image, 34 k-groups, whole iterations
  trunk_alloc(b, 0, P, &d->t, false);
  d->sh = b.f(P * 128); d->sig = b.f(P);
  if (st_net) {
    d->refpl = b.f((long long)R * 6); d->refpe = b.f((long long)R * 66); d->reff = b.f((long long)R * kF);
    {  // x spill: bf16 tile image over view SLOTS (VP per point), padded to the kernels' 256-row iterations
      const long long slots = ((P * (V <= 8 ? 8 : 16) + 255) / 256) * 256;
      d->X = b.f(slots * 64);
    }
    d->vis2 = b.f(M); d->rd = b.f(M * 4); d->meff = b.f(M); d->rgbin = b.f(M * 3);
    d->ch = b.f((M > ((P + 255) / 256) * 256 ? M : ((P + 255) / 256) * 256) * 128); d->ch2 = b.f(M * 64); d->logit = b.f(M);
  } else {
    d->ptspe = b.f(P * 33); d->dirpe = b.f((long long)R * 27);
    d->G4h = b.f(P * 256); d->G4 = b.f(P * 128);
    d->ch = b.f(P * 128); d->ch2 = b.f(P * 64); d->rgb = b.f(P * 3);
  }
  return b.off;
}

size_t net_fused_workspace(int kind, int R, int S, int V) {
  Bump b{nullptr, 0};
  FusedBufs d;
  int rc = net_rows_per_chunk(S, V);
  return fused_alloc(b, kind == DYN_NET_STATIC, R < rc ? R : rc, S, V, &d);
}

// per-point stage on the fused chains: point1 (geometry_fc, Q|K|V) -> ray-transformer
// attention (tcgen05 when S divides 128, else the SIMT kernel) -> point2 (fc + LayerNorm + heads);
// G, Q, K, V, O are bf16 tile images, g2 / GW use the fp32 tile layout (fused_engine.cuh)
static int run_point_fused(const dyn_net* n, const float* G, long long P, int R, int S, bool dynamic,
                           float* posenc_tab, TrunkBufs& t, Point2Args& p2, cudaStream_t st) {
  Point1Args p1;
  memset(&p1, 0, sizeof(p1));
  // Q, K, V, O travel between the point kernels as bf16 rows (they are tensor-core operands)
  __nv_bfloat16* Qb = reinterpret_cast<__nv_bfloat16*>(t.Q);
  __nv_bfloat16* Kb = reinterpret_cast<__nv_bfloat16*>(t.K);
  __nv_bfloat16* Vb = reinterpret_cast<__nv_bfloat16*>(t.V);
  __nv_bfloat16* Ob = reinterpret_cast<__nv_bfloat16*>(t.O);
  p1.G = G; p1.P = P; p1.S = S; p1.g2 = t.G2; p1.Q = Qb; p1.K = Kb; p1.V = Vb;
  p1.posenc = nullptr;
  if (dynamic) {
    posenc_table_kernel<<<cdiv((long long)S * 128, 256), 256, 0, st>>>(posenc_tab, S);
    DYN_LAUNCH_CHECK();
    p1.posenc = posenc_tab;
  }
  RUN(launch_point1_twin(n, p1, st));
  if (attention_tc_supported(S)) {
    RUN(launch_attention_tc(Qb, Kb, Vb, t.nvalid, P, S, Ob, st));
  } else {
    int threads = ((S + 31) / 32) * 32;
    size_t smem = (size_t)2 * S * 32 * sizeof(float);
    if (threads > 1024) return fail(DYN_E_INVALID, "ray transformer supports S <= 1024 (got %d)", S);
    if (smem > 48 * 1024)
      DYN_CUDA(cudaFuncSetAttribute(attention_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    ProfScope prof(PROF_ATTENTION, st);
    attention_kernel<true><<<R, threads, smem, st>>>(Qb, Kb, Vb, t.nvalid, S, Ob);
    DYN_LAUNCH_CHECK();
  }
  p2.O = Ob; p2.g2 = t.G2; p2.nvalid = t.nvalid; p2.P = P; p2.S = S;
  return launch_point2_twin(n, p2, st);
}

// unit-test hook: the per-point fused stage on caller-provided G / nvalid
// fp32 rows -> bf16 tile image with KG k-groups (columns >= ncols are zero)
__global__ void rows_to_image_kernel(const float* __restrict__ src, int ld, int ncols, long long P, int KG,
                                     uint8_t* __restrict__ img) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P * KG) return;
  const long long row = e / KG;
  const int kg = (int)(e % KG);
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = (8 * kg + i < ncols) ? src[row * ld + 8 * kg + i] : 0.f;
  if (KG == 34 && kg == 33) { v[0] = 1.f; v[1] = 1.f; }  // bias columns of the geometry_fc layers (chains_twin.cu)
  *reinterpret_cast<uint4*>(img + fe::tile_image_off(row, kg, KG)) =
      make_uint4(fe::pack_bf16x2(v[0], v[1]), fe::pack_bf16x2(v[2], v[3]), fe::pack_bf16x2(v[4], v[5]),
                 fe::pack_bf16x2(v[6], v[7]));
}
// fp32 tile layout (tile_f32_off) -> fp32 rows [P,128]
__global__ void tile_f32_to_rows_kernel(const uint8_t* __restrict__ src, long long P, float* __restrict__ dst) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P * 32) return;
  const long long row = e >> 5;
  const int cg = (int)(e & 31);
  reinterpret_cast<float4*>(dst)[row * 32 + cg] = *reinterpret_cast<const float4*>(src + fe::tile_f32_off(row, cg));
}

// Unit-test hook: plain fp32 rows in and out; the tile layouts the fused kernels exchange are
// converted here (scratch is allocated per call: this entry point is not on the product path).
// The Q, K, V, O arguments are ignored (those intermediates live in tile-image scratch).
int debug_point_chain(const dyn_net* n, const float* G, const float* nvalid, const float* pts,
                      const float* ray_dir, int R, int S, float* g2, float* Q, float* K, float* V,
                      float* O, float* out_a, float* out_b, float* posenc_ws, cudaStream_t st) {
  (void)Q; (void)K; (void)V; (void)O;
  const long long P = (long long)R * S;
  if (P == 0) return DYN_OK;
  const long long Pt = ((P + 255) / 256) * 256;
  const size_t g_bytes = fe::tile_image_bytes(Pt, 34), t_bytes = (size_t)Pt * 512;
  uint8_t* scratch = nullptr;
  DYN_CUDA(cudaMalloc(&scratch, g_bytes + 6 * t_bytes));
  DYN_CUDA(cudaMemsetAsync(scratch, 0, g_bytes + 6 * t_bytes, st));
  uint8_t* gimg = scratch;
  float* buf[6];
  for (int i = 0; i < 6; ++i) buf[i] = reinterpret_cast<float*>(scratch + g_bytes + (size_t)i * t_bytes);
  rows_to_image_kernel<<<cdiv(P * 34, 256), 256, 0, st>>>(G, kGStride, 257, P, 34, gimg);
  TrunkBufs t;
  memset(&t, 0, sizeof(t));
  t.G2 = buf[0]; t.Q = buf[1]; t.K = buf[2]; t.V = buf[3]; t.O = buf[4]; t.nvalid = const_cast<float*>(nvalid);
  Point2Args p2;
  memset(&p2, 0, sizeof(p2));
  const bool dynamic = n->kind == DYN_NET_DYNAMIC;
  if (dynamic) { p2.pts = pts; p2.ray_dir = ray_dir; p2.raw = out_a; }
  else { p2.GW = buf[5]; p2.sigma = out_b; }
  int rc = run_point_fused(n, reinterpret_cast<const float*>(gimg), P, R, S, dynamic, posenc_ws, t, p2, st);
  if (rc == DYN_OK) {
    tile_f32_to_rows_kernel<<<cdiv(P * 32, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(buf[0]), P, g2);
    if (!dynamic)
      tile_f32_to_rows_kernel<<<cdiv(P * 32, 256), 256, 0, st>>>(reinterpret_cast<const uint8_t*>(buf[5]), P, out_a);
  }
  cudaStreamSynchronize(st);
  cudaFree(scratch);
  return rc;
}

static int fill_view_args(ViewFusedArgs* a, const float* query_cam, const float* src_rgbs,
                          const float* src_cams, const void* feat_cl, int V, int S, int H, int W,
                          int h, int w, cudaStream_t st) {
  memset(a, 0, sizeof(*a));
  RUN(build_view_cams(src_cams, V, query_cam, st, &a->cams));
  a->h_img = a->cams.h_img; a->w_img = a->cams.w_img;
  a->rgba = src_rgbs; a->feat_bf = reinterpret_cast<const uint16_t*>(feat_cl);
  a->H = H; a->W = W; a->h = h; a->w = w; a->V = V; a->S = S;
  return DYN_OK;
}

int net_static_fused(const dyn_net* n, const float* pts, const float* ray_o, const float* ray_d,
                     const float* query_cam, const float* src_rgbs, const float* src_cams,
                     const void* feat_cl, int R_all, int S, int V, int H, int W, int h, int w,
                     float* raw, float* mask_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  const StaticLayout& L = n->sl;
  const int prec = DYN_PREC_BF16;
  ViewFusedArgs va{};
  RUN(fill_view_args(&va, query_cam, src_rgbs, src_cams, feat_cl, V, S, H, W, h, w, st));
  const int RC = net_rows_per_chunk(S, V);
  for (int r0 = 0; r0 < R_all; r0 += RC) {
    const int R = (R_all - r0) < RC ? (R_all - r0) : RC;
    const long long P = (long long)R * S, M = P * V, p0 = (long long)r0 * S;
    Bump b{(char*)ws, 0};
    FusedBufs d;
    if (fused_alloc(b, true, R, S, V, &d) > ws_bytes)
      return fail(DYN_E_WORKSPACE, "net_static_fused: workspace %zu < %zu", ws_bytes, b.off);
    // per-ray reference feature: ref_feature_fc(PE(plucker(ray)))  (mlp_network.py:434,450)
    RUN(dyn_plucker_ref(ray_o + (long long)r0 * 3, ray_d + (long long)r0 * 3, R, d.refpl, st));
    RUN(launch_pe(d.refpl, 6, 6, 0, 0.f, 5, false, R, d.refpe, st));
    RUN(launch_linear(L1(n, L.ref_feat, d.refpe, d.reff, R, ACT_NONE), st));
    va.pts = pts + p0 * 3; va.pts_seq = nullptr; va.P = P;
    va.ref_feat = d.reff; va.dfeat = nullptr;
    va.G = d.G; va.nvalid = d.t.nvalid; va.mask_proj = mask_out + p0 * V; va.mask_eff = d.meff;
    va.X = d.X; va.vis2 = d.vis2; va.ray_diff = d.rd; va.rgb_in = d.rgbin;
    va.dbg = view_dbg_ptr();
    RUN(launch_view_fused(n, va, V, st));
    {
      Point2Args p2;
      memset(&p2, 0, sizeof(p2));
      p2.GW = d.ch;  // [P,128] (the staged head's scratch is free on this path)
      p2.sigma = d.sig;
      RUN(run_point_fused(n, d.G, P, R, S, false, nullptr, d.t, p2, st));
      RgbHeadArgs rh;
      memset(&rh, 0, sizeof(rh));
      rh.X = d.X; rh.vis2 = d.vis2; rh.ray_diff = d.rd; rh.mask_eff = d.meff; rh.rgb_in = d.rgbin;
      rh.GW = d.ch; rh.sigma = d.sig; rh.P = P; rh.V = V; rh.raw = raw + p0 * 4;
      RUN(launch_rgbhead_twin(n, rh, st));
    }
    (void)prec; (void)M;
  }
  return DYN_OK;
}

int net_dynamic_fused(const dyn_net* n, const float* pts, const float* pts_seq, const float* ray_dir,
                      const float* query_cam, const float* src_rgbs, const float* src_cams,
                      const void* feat_cl, float time, int R_all, int S, int V, int H, int W, int h,
                      int w, float* raw, float* mask_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  const DynamicLayout& L = n->dl;
  const int prec = DYN_PREC_BF16;
  ViewFusedArgs va{};
  RUN(fill_view_args(&va, query_cam, src_rgbs, src_cams, feat_cl, V, S, H, W, h, w, st));
  const long long P_all = (long long)R_all * S;
  const int RC = net_rows_per_chunk(S, V);
  for (int r0 = 0; r0 < R_all; r0 += RC) {
    const int R = (R_all - r0) < RC ? (R_all - r0) : RC;
    const long long P = (long long)R * S, p0 = (long long)r0 * S;
    Bump b{(char*)ws, 0};
    FusedBufs d;
    if (fused_alloc(b, false, R, S, V, &d) > ws_bytes)
      return fail(DYN_E_WORKSPACE, "net_dynamic_fused: workspace %zu < %zu", ws_bytes, b.off);
    dyn_time_feat_kernel<<<1, 256, 0, st>>>(n->params, L, time, d.small, 0);
    DYN_LAUNCH_CHECK();
    va.pts = pts + p0 * 3; va.pts_seq = pts_seq + p0 * 3; va.seq_stride = P_all; va.P = P;
    va.ref_feat = nullptr; va.dfeat = d.small;
    va.G = d.G; va.nvalid = d.t.nvalid; va.mask_proj = mask_out + p0 * V; va.mask_eff = nullptr;
    va.X = nullptr; va.vis2 = nullptr; va.ray_diff = nullptr; va.rgb_in = nullptr;
    RUN(launch_view_fused(n, va, V, st));
    {
      Point2Args p2;
      memset(&p2, 0, sizeof(p2));
      p2.pts = pts + p0 * 3; p2.ray_dir = ray_dir + (long long)r0 * 3; p2.raw = raw + p0 * 4;
      RUN(run_point_fused(n, d.G, P, R, S, true, d.G4h, d.t, p2, st));
    }
    (void)prec;
  }
  return DYN_OK;
}

int zero_last_samples(float* coeff, int R, int S, int width, cudaStream_t st) {
  int n_last = (int)lrint((double)S * 0.1);  // int(round(S*0.1)), render_ray.py:459 (banker's == Python round)
  if (n_last <= 0) n_last = S;  // Python's x[:, -0:, :] is the WHOLE axis
  if (R == 0) return DYN_OK;
  long long tot = (long long)R * n_last * width;
  zero_last_kernel<<<cdiv(tot, 256), 256, 0, st>>>(coeff, R, S, n_last, width);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // namespace dyn
