// Fused per-(point, view) stage of the two aggregation networks on tcgen05 (reference:
// ibrnet/projection.py:103-176, ibrnet/mlp_network.py:236-284 (dynamic) / :423-497 (static)).
// Per 128-row tile, without leaving the SM:
//
//   projection + in-front/in-bounds masks + view-angle difference   (a4, a6)
//   bilinear gather of source RGB + features from L2-resident maps  (a5)
//   [static]  Plucker coords, positional encodings, ray_dir_fc     (a7, a8, a10)
//   pooling weights, weighted mean/var over views (warp shuffles)  (a9/a10)
//   base_fc -> vis_fc -> vis_fc2 (tensor cores, fp32 accum in TMEM)
//   visibility re-weighting and the second mean/var pooling -> G (bf16 tile image) per point
//
// Engine: fused_engine.cuh (operand tile in shared memory written by the epilogues, accumulators
// in TMEM, weights streamed through a cp.async.bulk ring, table-driven MMA issuer).  Every row is
// served by TWO threads in twin warps w and w + 4 (same TMEM lane quadrant), which is what the
// latency-bound epilogues need; each twin owns half of every layer's output columns and half of the
// gathered / pooled channels, and the twins exchange only two scalars per row and iteration (the
// partial visibility logits).
//
// TWO independent CTAs per SM, each with one 128-row tile and a 2-slot weight ring, so the tensor pipe
// is shared by two unsynchronised instruction streams:
//   warps 0-3 : twin 0 (quadrant = w & 3)      warps 4-7 : twin 1 of the same rows
//   warp 8    : MMA issuer (one elected lane)  warp 9    : weight producer
//
// Every layer from base_fc.0 on is issued in two sub-rounds, so the tensor cores start on the finished
// operand columns while the row warps are still in the epilogue of the others (details at "From here on").
// The operand barriers count WARPS, not threads (warp_arrive).  The accumulator read-outs are
// software-pipelined in 16-column halves (fused_engine.cuh: tmem_pipe16).
//
// Latency hiding inside a CTA (round 2, profiles/r02_view_kernels.md): the source views are read in
// their packed per-frame layouts (bf16 channels-last features: 2 x 16-byte loads per tap and twin; RGBA
// fp32 images: 1 load per tap), the taps are ISSUED right after the projection and consumed after the
// positional-encoding operand has been built and handed to the tensor cores, the per-ray reference
// feature is loaded before the wait for ray_dir_fc.2, the next iteration's points before the last wait,
// and the camera matrices sit in shared memory (lanes of a warp index different views).
#include <cstdlib>
#include "fused_engine.cuh"
#include "geometry.cuh"
#include "nets.cuh"

namespace dyn {

using namespace tc;
using namespace fe;

namespace {

constexpr int kTwinATile = 69632;  // K <= 256 (+ one k-step of bias columns): 34 k-groups
// T_B5 / T_B7 hold log2(e) * bias, T_W6V / T_W8 hold ln(2) * weight (the hidden activations of vis_fc.0 and
// vis_fc2.0 live on the exp2 scale); the biases of base_fc.2 and vis_fc.2 ride in the MMA
constexpr int T_B2 = 0, T_B5 = 48, T_W6V = 176, T_B7 = 304, T_W8 = 432, T_MISC = 560, T_DFEAT = 576,
              T_CAMS = 624 /* 16 views x (P 12 + centre 3 + pad) */, T_XCH = T_CAMS + 256;  // + 2 x [2][128] exchange
constexpr int kTwinConst = T_XCH + 512;
// weight ring: 16 KB stages; 8 KB stages x twice the slots measured 14 % slower (per-chunk barrier and
// issue overhead outweighs the faster slot turnover, profiles/r01_kernels.md)
constexpr int kTwinStage = 16384;
constexpr int kTwinRing = 2;
constexpr int kTwinSmem = kTwinATile + kTwinRing * kTwinStage + kTwinConst * 4 + 256;

__device__ __forceinline__ void pair_sync(int pair) {
  asm volatile("bar.sync %0, 64;" ::"r"(pair + 1) : "memory");
}

// One arrival per warp on an operand barrier: every thread has fenced its own writes (fence.proxy.async +
// tcgen05.fence::before_thread_sync), the warp converges (__syncwarp orders the lanes' memory operations) and
// lane 0 arrives once -- 32 same-address shared-memory atomics per warp instruction become one
__device__ __forceinline__ void warp_arrive(uint32_t bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}

// 11 values of one PE component: [x, cos(2^k x) k=0..4, sin(2^k x) k=0..4]
__device__ __forceinline__ void pe_comp(float x, float* o) {
  float s, c;
  __sincosf(x, &s, &c);
  o[0] = x;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    o[1 + k] = c;
    o[6 + k] = s;
    const float s2 = 2.f * s * c, c2 = 1.f - 2.f * s * s;
    s = s2; c = c2;
  }
}

template <int VP, bool ST>
__global__ void __launch_bounds__(320, 2) view_twin3_kernel(const __grid_constant__ ViewFusedArgs a) {
  constexpr int ROWS = 128;  // rows per iteration: one tile
  constexpr int W_ISSUE = 8, W_PROD = 9;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem + kTwinATile;
  float* cst = reinterpret_cast<float*>(ring + kTwinRing * kTwinStage);
  uint64_t* bars = reinterpret_cast<uint64_t*>(cst + kTwinConst);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  __shared__ __align__(16) FusedChunk s_tab[kMaxChunks];
  stage_chunks(s_tab, a.chunks, a.nchunks);

  if (tid == 0) {
    init_barriers(bar0, /*pp=*/false, /*arrivals=*/128, kTwinRing);
    // both operand barriers count one arrival per row warp (warp_arrive); the second one serves sub-round 1
    // of the pipelined layers
    mbar_init(bar_aready(bar0, 1, kTwinRing), 8);
    mbar_init(bar_aready(bar0, 0, kTwinRing), 8);
    mbar_fence_init();
  }
  {
    const float* prm = a.params;
    for (int i = tid; i < 256; i += blockDim.x) {  // camera matrices: lanes index them by view
      const int vv = i >> 4, j = i & 15;
      cst[T_CAMS + i] = j < 12 ? a.cams.P[vv][j] : (j < 15 ? a.cams.center[vv][j - 12] : 0.f);
    }
    for (int i = tid; i < 128; i += blockDim.x) {
      cst[T_B5 + i] = prm[a.o_b5 + i] * 1.4426950408889634f;
      cst[T_W6V + i] = prm[a.o_w6 + 128 * 128 + i] * 0.6931471805599453f;
      cst[T_B7 + i] = prm[a.o_b7 + i] * 1.4426950408889634f;
      cst[T_W8 + i] = prm[a.o_w8 + i] * 0.6931471805599453f;
    }
    if (tid < 48) cst[T_B2 + tid] = (ST && tid < kF) ? prm[a.o_b2 + tid] : 0.f;
    if (tid < 40) cst[T_DFEAT + tid] = (!ST && tid < kF) ? a.dfeat[tid] : 0.f;
    if (tid == 0) {
      cst[T_MISC + 0] = prm[a.o_b6 + 128];
      cst[T_MISC + 1] = prm[a.o_b8];
      cst[T_MISC + 2] = (ST && a.o_s >= 0) ? fabsf(prm[a.o_s]) : 0.f;
    }
  }
  if (warp == W_ISSUE) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const long long n_rows = a.P * VP;
  const int n_iter = (int)((n_rows + ROWS - 1) / ROWS);

  if (warp == W_PROD) {
    if ((tid & 31) < a.producers)
      producer_loop<false, kTwinRing, kTwinStage>(s_tab, a.nchunks, a.wimg, n_iter, ring, bar0, tid & 31, a.producers);
  } else if (warp == W_ISSUE) {
    issuer_loop<false, 1, kTwinRing, kTwinStage>(s_tab, a.nchunks, n_iter, smem, ring, bar0, tmem_base, kTwinATile,
                                                  a.dbg ? a.dbg + 128 : nullptr);
  } else {
    const int tw = tid / ROWS;         // twin index
    const int t = tid % ROWS;          // row inside the tile
    uint8_t* arow = smem + (t >> 3) * 128 + (t & 7) * 16;
    const uint32_t tacc = tmem_addr(tmem_base, (uint32_t)((warp & 3) * 32), 0u);
    const int v = t % VP;
    const int gl = t & (VP - 1);
    const int pair = warp & 3;
    const uint32_t a_ready = bar_aready(bar0, 0, kTwinRing), acc_full = bar_acc(bar0, 0, kTwinRing);
    float* xch5 = cst + T_XCH;        // [2][128] partial visibility logits of vis_fc
    float* xch7 = cst + T_XCH + 256;  // [2][128] partial logits of vis_fc2
    if (tw == 0) {
      // persistent bias columns of base_fc.2 (K = 256 + 16): k-groups 32, 33 = [1, 1, 0 ...] (hi, lo)
      float o[8] = {1.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      store8(arow, 256, o);
      store8(arow, 264, z);
    }
    uint32_t acc_cnt = 0;
    const float wh = a.w_img, hh = a.h_img;
    int dbg_n = 0;
#define TS()                                                                            \
  do {                                                                                  \
    if (a.dbg != nullptr && blockIdx.x == 0 && t == 0 && dbg_n < 64)                 \
      a.dbg[tw * 64 + dbg_n++] = clock64();                                             \
  } while (0)

    // the first point of this thread; later ones are fetched one iteration ahead (before the last MMA wait)
    float np3[3], nq3[3];
    auto fetch_point = [&](int it2) {
      const long long pl2 = ((long long)it2 * ROWS + t) / VP;
      np3[0] = 0.f; np3[1] = 0.f; np3[2] = 0.f;
      if (pl2 < a.P) { np3[0] = a.pts[pl2 * 3]; np3[1] = a.pts[pl2 * 3 + 1]; np3[2] = a.pts[pl2 * 3 + 2]; }
      nq3[0] = np3[0]; nq3[1] = np3[1]; nq3[2] = np3[2];
      if (!ST && pl2 < a.P && v < a.V) {
        const float* q = a.pts_seq + ((long long)v * a.seq_stride + pl2) * 3;
        nq3[0] = q[0]; nq3[1] = q[1]; nq3[2] = q[2];
      }
    };
    if ((int)blockIdx.x < n_iter) fetch_point((int)blockIdx.x);
    const bool want_rgb = (tw == 0) || (ST && a.mask_rgb);

    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      const long long pl = ((long long)it * ROWS + t) / VP;
      const bool pt_ok = pl < a.P;
      const bool valid = pt_ok && v < a.V;
      const long long m = pl * a.V + v;
      const long long ray = pt_ok ? pl / a.S : 0;

      TS();  // 0: iteration start
      // ---- geometry (both twins; cheap) ----
      const float p3[3] = {np3[0], np3[1], np3[2]}, q3[3] = {nq3[0], nq3[1], nq3[2]};
      const int vc = valid ? v : 0;
      const float* cam = cst + T_CAMS + 16 * vc;  // P (12) | centre (3)
      float pu, pv;
      bool front;
      project_point(cam, q3[0], q3[1], q3[2], pu, pv, front);
      const bool inb = (pu <= wh - 1.f) && (pu >= 0.f) && (pv <= hh - 1.f) && (pv >= 0.f);
      const float mask_proj = (valid && inb && front) ? 1.f : 0.f;

      // ---- issue the bilinear taps now: 2 x 16 B per tap of this twin's 16 bf16 feature channels
      //      (+ 1 x 16 B RGBA); they are consumed after the ray_dir_fc.0 operand has been built ----
      uint4 tf[8];
      float4 tr[4];
      float tw4[4], twr[4];
      {
        const float gx = 2.f * pu / (wh - 1.f) - 1.f, gy = 2.f * pv / (hh - 1.f) - 1.f;
        const bool ld = valid && !(a.ablate & 1);
        {
          const float fx = (gx + 1.f) * 0.5f * (float)(a.w - 1), fy = (gy + 1.f) * 0.5f * (float)(a.h - 1);
          const float x0f = floorf(fx), y0f = floorf(fy);
          const int x0 = (int)x0f, y0 = (int)y0f;
          const float ax = fx - x0f, ay = fy - y0f, bx = (x0f + 1.f) - fx, by = (y0f + 1.f) - fy;
          const uint16_t* base = a.feat_bf + (long long)vc * a.h * a.w * kC + 16 * tw;
#pragma unroll
          for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
              // out-of-range taps (and padding rows) load a clamped texel with weight 0: no branch, all loads
              // of this thread are in flight together
              const int xi = x0 + dx, yi = y0 + dy;
              const bool in = ld && xi >= 0 && xi < a.w && yi >= 0 && yi < a.h;
              tw4[2 * dy + dx] = in ? (dx ? ax : bx) * (dy ? ay : by) : 0.f;
              const int xc = min(max(xi, 0), a.w - 1), yc = min(max(yi, 0), a.h - 1);
              const uint4* tp = reinterpret_cast<const uint4*>(base + ((long long)yc * a.w + xc) * kC);
              tf[2 * (2 * dy + dx)] = __ldg(tp);
              tf[2 * (2 * dy + dx) + 1] = __ldg(tp + 1);
            }
        }
        if (want_rgb) {
          const float fx = (gx + 1.f) * 0.5f * (float)(a.W - 1), fy = (gy + 1.f) * 0.5f * (float)(a.H - 1);
          const float x0f = floorf(fx), y0f = floorf(fy);
          const int x0 = (int)x0f, y0 = (int)y0f;
          const float ax = fx - x0f, ay = fy - y0f, bx = (x0f + 1.f) - fx, by = (y0f + 1.f) - fy;
          const float* base = a.rgba + (long long)vc * a.H * a.W * 4;
#pragma unroll
          for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
              const int xi = x0 + dx, yi = y0 + dy;
              const bool in = ld && xi >= 0 && xi < a.W && yi >= 0 && yi < a.H;
              twr[2 * dy + dx] = in ? (dx ? ax : bx) * (dy ? ay : by) : 0.f;
              const int xc = min(max(xi, 0), a.W - 1), yc = min(max(yi, 0), a.H - 1);
              tr[2 * dy + dx] = __ldg(reinterpret_cast<const float4*>(base + ((long long)yc * a.W + xc) * 4));
            }
        }
      }

      float rd[4];
      {
        float a0 = a.cams.tgt[0] - p3[0], a1 = a.cams.tgt[1] - p3[1], a2 = a.cams.tgt[2] - p3[2];
        normalize3(a0, a1, a2);
        float b0 = cam[12] - q3[0], b1 = cam[13] - q3[1], b2 = cam[14] - q3[2];
        normalize3(b0, b1, b2);
        rd[0] = a0 - b0; rd[1] = a1 - b1; rd[2] = a2 - b2;
        rd[3] = a0 * b0 + a1 * b1 + a2 * b2;
        normalize3(rd[0], rd[1], rd[2]);
      }

      if (ST) {
        // ---- layer-1 operand, 56 columns per twin (component-major PE, see view_twin3_build); each
        //      8-column group is stored as soon as it is complete (short register live ranges while the
        //      taps are in flight).  Padding rows keep (finite) garbage: every use of their layer outputs
        //      is guarded by `valid` ----
        float pl6[6];
        {
          const float ox = cam[12], oy = cam[13], oz = cam[14];
          float dx = p3[0] - ox, dy = p3[1] - oy, dz = p3[2] - oz;
          normalize3(dx, dy, dz);
          pl6[0] = dx; pl6[1] = dy; pl6[2] = dz;
          pl6[3] = oy * dz - oz * dy;
          pl6[4] = oz * dx - ox * dz;
          pl6[5] = ox * dy - oy * dx;
        }
        float xin[56];
        if (tw == 0) {
          pe_comp(p3[0], xin);         store8(arow, 0, xin);
          pe_comp(p3[1], xin + 11);    store8(arow, 8, xin + 8);
          pe_comp(p3[2], xin + 22);    store8(arow, 16, xin + 16); store8(arow, 24, xin + 24);
          pe_comp(pl6[0], xin + 33);   store8(arow, 32, xin + 32);
          pe_comp(pl6[1], xin + 44);   xin[55] = 0.f;
          store8(arow, 40, xin + 40);  store8(arow, 48, xin + 48);
        } else {
          pe_comp(pl6[2], xin);        store8(arow, 56, xin);
          pe_comp(pl6[3], xin + 11);   store8(arow, 64, xin + 8);
          pe_comp(pl6[4], xin + 22);   store8(arow, 72, xin + 16); store8(arow, 80, xin + 24);
          pe_comp(pl6[5], xin + 33);   store8(arow, 88, xin + 32);
          xin[44] = rd[0]; xin[45] = rd[1]; xin[46] = rd[2]; xin[47] = rd[3];
          xin[48] = 1.f; xin[49] = 1.f;  // bias columns of ray_dir_fc.0 (hi, lo)
#pragma unroll
          for (int i = 50; i < 56; ++i) xin[i] = 0.f;
          store8(arow, 96, xin + 40);  store8(arow, 104, xin + 48);
        }
        fence_proxy_async_smem();
        tc_fence_before_sync();
        warp_arrive(a_ready);
      }

      TS();  // 1: after F1 operand + arrive
      // ---- consume the taps: rgb (twin 0, or both when mask_rgb) + this twin's 16 feature channels ----
      float chv[40];  // this twin's pooled channels (layout in view_twin3_build)
#pragma unroll
      for (int i = 0; i < 40; ++i) chv[i] = 0.f;
      float rgb[3] = {0.f, 0.f, 0.f};
      {
#pragma unroll
        for (int tp = 0; tp < 4; ++tp) {
          const float wgt = tw4[tp];
#pragma unroll
          for (int hlf = 0; hlf < 2; ++hlf) {
            const uint4 q = tf[2 * tp + hlf];
            const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float lo = __uint_as_float(u[j] << 16), hi = __uint_as_float(u[j] & 0xffff0000u);
              if (tw == 0) {
                chv[3 + 8 * hlf + 2 * j] += lo * wgt; chv[3 + 8 * hlf + 2 * j + 1] += hi * wgt;
              } else {
                chv[8 * hlf + 2 * j] += lo * wgt; chv[8 * hlf + 2 * j + 1] += hi * wgt;
              }
            }
          }
        }
        if (want_rgb) {
#pragma unroll
          for (int tp = 0; tp < 4; ++tp) {
            rgb[0] += tr[tp].x * twr[tp]; rgb[1] += tr[tp].y * twr[tp]; rgb[2] += tr[tp].z * twr[tp];
          }
        }
      }
      float mask = mask_proj;
      if (ST && a.mask_rgb) mask *= ((rgb[0] + rgb[1] + rgb[2]) > 1e-3f) ? 1.f : 0.f;
      if (tw == 0) {
        chv[0] = rgb[0]; chv[1] = rgb[1]; chv[2] = rgb[2];
        if (valid && !(a.ablate & 2)) {
          a.mask_proj[m] = mask_proj;
          if (ST) {
            a.mask_eff[m] = mask;
            reinterpret_cast<float4*>(a.ray_diff)[m] = make_float4(rd[0], rd[1], rd[2], rd[3]);
            a.rgb_in[m * 3] = rgb[0]; a.rgb_in[m * 3 + 1] = rgb[1]; a.rgb_in[m * 3 + 2] = rgb[2];
          }
        }
      }

      TS();  // 2: after gather
      if (ST) {
        // ---- F1 epilogue: this twin's 128 of the 256 columns ----
        mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
        TS();  // 3: F1 acc ready
        tc_fence_after_sync();
        tmem_pipe16<8>(tacc, [&](int h) { return 128 * tw + 16 * h; }, [&](int h, float* v) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = elu_log2(v[i]);
          store8(arow, 128 * tw + 16 * h, v);
          store8(arow, 128 * tw + 16 * h + 8, v + 8);
        });
        fence_proxy_async_smem();
        tc_fence_before_sync();
        warp_arrive(a_ready);
        TS();  // 4: F1 epilogue done
        // ---- F2: src_feat (35 of 48 columns) * ref_feat; twin 0 keeps 0..17, twin 1 keeps 18..34.
        //      The per-ray reference feature is loaded BEFORE the wait (its L2 latency hides behind the MMA) ----
        float rfv[18];
        {
          const float* rf = a.ref_feat + ray * kF + 18 * tw;
#pragma unroll
          for (int i = 0; i < 18; ++i) rfv[i] = (tw == 0 || i < 17) ? __ldg(rf + i) : 0.f;
        }
        mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
        TS();  // 5: F2 acc ready
        tc_fence_after_sync();
        float s48[48];
        tmem_ld32(tacc, s48);
        tmem_ld16(tacc + 32, s48 + 32);
        tmem_wait_ld();
        if (tw == 0) {
#pragma unroll
          for (int i = 0; i < 18; ++i) chv[19 + i] = valid ? (s48[i] + cst[T_B2 + i]) * rfv[i] : 0.f;
        } else {
#pragma unroll
          for (int i = 0; i < 17; ++i)
            chv[16 + i] = valid ? (s48[18 + i] + cst[T_B2 + 18 + i]) * rfv[i] : 0.f;
        }
      } else {
        // dynamic: + time feature on this twin's channels (mlp_network.py:244-247)
        if (tw == 0) {
#pragma unroll
          for (int i = 0; i < 19; ++i) chv[i] = valid ? chv[i] + cst[T_DFEAT + i] : 0.f;
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) chv[i] = valid ? chv[i] + cst[T_DFEAT + 19 + i] : 0.f;
        }
      }

      // ---- pooling weights (both twins) ----
      float w1;
      if (ST && a.anti_alias) {
        const float e = ex2f(cst[T_MISC + 2] * (rd[3] - 1.f) * 1.4426950408889634f);
        const float emin = group_min<VP>(valid ? e : INFINITY);
        w1 = valid ? (e - emin) * mask : 0.f;
      } else {
        w1 = mask;
      }
      w1 = w1 / (group_sum<VP>(w1) + 1e-8f);

      // ---- first pooling on this twin's channel groups: [mean8 | var8 | feat8] per group.  Static net: twin 0 at
      //      columns [0,120), twin 1 at [128,248) (K = 256); after three of the five groups both twins arrive once
      //      so that the first half of base_fc.0 (k-steps 0-3 and 8-11) runs while the last two groups are pooled ----
      {
        constexpr int ng0 = ST ? 5 : 3, ng1 = ST ? 5 : 2;
        const int col_base = tw == 0 ? 0 : (ST ? 128 : 24 * ng0);
#pragma unroll
        for (int g = 0; g < ng0; ++g) {
          if (tw == 1 && g >= ng1) break;
          float o[24];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float fv = chv[8 * g + j];
            const float s1 = group_sum<VP>(w1 * fv);
            const float d = fv - s1;
            const float s2 = group_sum<VP>(w1 * d * d);
            o[j] = s1; o[8 + j] = s2; o[16 + j] = fv;
          }
          // bias columns of base_fc.0 (hi, lo): the last (unused) channel slot of twin 0
          if (tw == 0 && g == ng0 - 1) { o[7] = 1.f; o[15] = 1.f; }
          store8(arow, col_base + 24 * g, o);
          store8(arow, col_base + 24 * g + 8, o + 8);
          store8(arow, col_base + 24 * g + 16, o + 16);
          if (ST && g == 2) {
            fence_proxy_async_smem();
            tc_fence_before_sync();
            warp_arrive(a_ready);
          }
        }
        {  // zero the K padding (static: 120..127 / 248..255, dynamic: 120..127)
          float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
          if (ST) store8(arow, 120 + 128 * tw, z);
          else if (tw == 1) store8(arow, 120, z);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      warp_arrive(bar_aready(bar0, ST ? 1 : 0, kTwinRing));  // static: sub-round 1 of base_fc.0 (second operand barrier)

      TS();  // 6: pool1 done + arrive
      // From here on every layer runs in TWO sub-rounds: the twins own interleaved 32-column blocks, arrive after
      // each block, and the issuer starts the next layer's k-steps over the finished columns while the other block
      // is still in its epilogue.  Accumulators alternate between TMEM columns [0,128) and [128,256); x lives as
      // bf16 in operand columns [0,128) (vis_fc.0 reads it there, vis_fc.2 adds to it), h in [128,256).
      // ---- F3: ELU(base_fc.0): this twin's blocks 4+tw, 6+tw (columns 128..255 first: they free the TMEM half
      //      base_fc.2 accumulates into), then 0+tw, 2+tw ----
      mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
      TS();  // 7: F3 acc ready
      tc_fence_after_sync();
      {
        auto col3 = [&](int h) { const int j = h >> 1; return 32 * ((j < 2 ? 4 : 0) + 2 * (j & 1) + tw) + 16 * (h & 1); };
        tmem_pipe16<8>(tacc, col3, [&](int h, float* v) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = elu_log2(v[i]);
          store8(arow, col3(h), v);
          store8(arow, col3(h) + 8, v + 8);
          if ((h & 3) == 3) {
            fence_proxy_async_smem();
            tc_fence_before_sync();
            warp_arrive(bar_aready(bar0, h >> 2, kTwinRing));  // first / second operand barrier
          }
        });
      }

      TS();  // 8: F3 epilogue done
      // ---- F4: x = ELU(base_fc.2) (accumulator in TMEM [128,256), bias folded, exp2 scale) -> bf16 operand
      //      columns of this twin's blocks tw, 2 + tw (the pooling weight w1 of vis_fc.0's input is applied to
      //      that layer's accumulator: W (w1 x) = w1 (W x)) ----
      mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
      TS();  // 9: F4 acc ready
      tc_fence_after_sync();
      auto colh = [&](int h) { return 32 * (2 * (h >> 1) + tw) + 16 * (h & 1); };  // this twin's blocks tw, 2 + tw
      tmem_pipe16<4>(tacc + 128, colh, [&](int h, float* v) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = elu_from_log2(v[i]);
        store8(arow, colh(h), v);
        store8(arow, colh(h) + 8, v + 8);
        if (h & 1) {
          fence_proxy_async_smem();
          tc_fence_before_sync();
          warp_arrive(bar_aready(bar0, h >> 1, kTwinRing));
        }
      });

      TS();  // 10: F4 epilogue done
      // ---- F5: h = ELU(w1 (vis_fc.0 x) + b) -> operand columns [128,256); partial visibility logit ----
      mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
      TS();  // 11: F5 acc ready
      tc_fence_after_sync();
      {
        float part = 0.f;
        tmem_pipe16<4>(tacc, colh, [&](int h, float* v) {
          const int c0 = colh(h);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            v[i] = elu_log2(fmaf(v[i], w1, cst[T_B5 + c0 + i]));  // log2(e) * ELU(w1 (W x) + b)
            part = fmaf(v[i], cst[T_W6V + c0 + i], part);
          }
          store8(arow, 128 + c0, v);
          store8(arow, 128 + c0 + 8, v + 8);
          if (h & 1) {
            if (h == 3) xch5[tw * 128 + t] = part;
            fence_proxy_async_smem();
            tc_fence_before_sync();
            warp_arrive(bar_aready(bar0, h >> 1, kTwinRing));
          }
        });
      }

      TS();  // 12: F5 epilogue done
      // ---- F6: x += ELU(vis_fc.2[:128] h) (accumulator in TMEM [128,256), bias folded); bf16(x) is vis_fc2.0's
      //      operand (vis1 is applied to its accumulator) and, for the static net, the blending head's input ----
      mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
      TS();  // 13: F6 acc ready
      tc_fence_after_sync();
      // both twins arrived on a_ready before this MMA ran: the partial logits are visible
      const float vlogit = cst[T_MISC + 0] + xch5[t] + xch5[128 + t];
      const float vis1 = sigmoid_fast(elu_fast(vlogit)) * mask;
      tmem_pipe16<4>(tacc + 128, colh, [&](int h, float* v) {
        const int c0 = colh(h);
        uint4 pk[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const uint4 q = *reinterpret_cast<const uint4*>(arow + ((c0 >> 3) + i) * 2048);
          const uint32_t u[4] = {q.x, q.y, q.z, q.w};
          uint32_t o[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float lo = __uint_as_float(u[k] << 16) + elu_from_log2(v[8 * i + 2 * k]);
            const float hi = __uint_as_float(u[k] & 0xffff0000u) + elu_from_log2(v[8 * i + 2 * k + 1]);
            o[k] = pack_bf16x2(lo, hi);
          }
          pk[i] = make_uint4(o[0], o[1], o[2], o[3]);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) *reinterpret_cast<uint4*>(arow + ((c0 >> 3) + i) * 2048) = pk[i];
        if (h & 1) {
          fence_proxy_async_smem();
          tc_fence_before_sync();
          warp_arrive(bar_aready(bar0, h >> 1, kTwinRing));
        }
        // static net: x is spilled as a bf16 tile image (fused_engine.cuh) in view-slot row order, which the
        // blending head lands in its operand tile with one bulk copy per 128 rows.  The global stores are issued
        // AFTER the operand barrier arrival (fence.proxy.async is a MEMBAR: it would wait for them to be performed)
        if (ST && !(a.ablate & 2)) {
          uint8_t* xo = reinterpret_cast<uint8_t*>(a.X) + tile_image_off((long long)it * ROWS + t, c0 >> 3, 16);
#pragma unroll
          for (int i = 0; i < 2; ++i) *reinterpret_cast<uint4*>(xo + i * 2048) = pk[i];
        }
      });

      TS();  // 14: F6 epilogue done
      if (it + (int)gridDim.x < n_iter) fetch_point(it + (int)gridDim.x);  // next iteration's point
      // ---- F7: vis2 = sigmoid(vis_fc2.2 . ELU(vis1 (vis_fc2.0 x) + b)) * mask ----
      mbar_wait(acc_full, acc_cnt & 1); ++acc_cnt;
      TS();  // 15: F7 acc ready
      tc_fence_after_sync();
      {
        float part = 0.f;
        tmem_pipe16<4>(tacc, colh, [&](int h, float* v) {
          const int c0 = colh(h);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            part = fmaf(elu_log2(fmaf(v[i], vis1, cst[T_B7 + c0 + i])), cst[T_W8 + c0 + i], part);
        });
        xch7[tw * 128 + t] = part;
      }
      TS();  // 16: F7 partial done
      pair_sync(pair);
      const float v2 = cst[T_MISC + 1] + xch7[t] + xch7[128 + t];
      const float vis2 = sigmoid_fast(v2) * mask;
      if (ST && valid && tw == 0 && !(a.ablate & 2)) a.vis2[m] = vis2;
      const float vsum = group_sum<VP>(vis2);
      const float w2 = vis2 / (vsum + 1e-8f);
      const float W = group_sum<VP>(w2);
      const float nval = group_sum<VP>(mask);

      // ---- second pooling on this twin's 64 channels (blocks tw and 2 + tw of bf16(x) in the operand tile):
      //      reduce-scatter of sum(w x), sum(w x^2) over the point's view lanes ----
      if (!(a.ablate & 8)) {
        const bool b0 = gl & 1, b1 = gl & 2, b2 = gl & 4, b3 = gl & 8;
        constexpr int NO = VP == 16 ? 4 : 8;
        const int cbase = 32 * ((b0 ? 2 : 0) + tw) + (b1 ? 16 : 0) + (b2 ? 8 : 0) + ((VP == 16 && b3) ? 4 : 0);
        float mean[NO], sq[NO];
        float lo[32], hi[32];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 ql = *reinterpret_cast<const uint4*>(arow + (4 * tw + i) * 2048);
          const uint4 qh = *reinterpret_cast<const uint4*>(arow + (8 + 4 * tw + i) * 2048);
          const uint32_t ul[4] = {ql.x, ql.y, ql.z, ql.w}, uh[4] = {qh.x, qh.y, qh.z, qh.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            lo[8 * i + 2 * k] = __uint_as_float(ul[k] << 16); lo[8 * i + 2 * k + 1] = __uint_as_float(ul[k] & 0xffff0000u);
            hi[8 * i + 2 * k] = __uint_as_float(uh[k] << 16); hi[8 * i + 2 * k + 1] = __uint_as_float(uh[k] & 0xffff0000u);
          }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float s1[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float l = q ? w2 * lo[i] * lo[i] : w2 * lo[i];
            const float h = q ? w2 * hi[i] * hi[i] : w2 * hi[i];
            const float send = b0 ? l : h, keep = b0 ? h : l;
            s1[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
          }
          float s2[16], s3[8];
          rs_step<32>(s1, s2, b1, 2);
          rs_step<16>(s2, s3, b2, 4);
          float* dst = q ? sq : mean;
          if (VP == 16) {
            float s4[4];
            rs_step<8>(s3, s4, b3, 8);
#pragma unroll
            for (int i = 0; i < NO; ++i) dst[i] = s4[i < 4 ? i : 0];
          } else {
#pragma unroll
            for (int i = 0; i < NO; ++i) dst[i] = s3[i < 8 ? i : 0];
          }
        }
        if (pt_ok && !(a.ablate & 4)) {
          // pooled statistics as the bf16 tile image of geometry_fc's operand (34 k-groups:
          // mean 0..127 | var 128..255 | weight 256 | zero pad), rows = points
          uint8_t* gi = reinterpret_cast<uint8_t*>(a.G);
          float mu[NO], vr[NO];
#pragma unroll
          for (int i = 0; i < NO; ++i) {
            mu[i] = mean[i];
            vr[i] = sq[i] - mu[i] * mu[i] * (2.f - W);
          }
          uint8_t* pm = gi + tile_image_off(pl, cbase >> 3, 34) + (cbase & 7) * 2;
          uint8_t* pv = gi + tile_image_off(pl, 16 + (cbase >> 3), 34) + (cbase & 7) * 2;
          if (NO == 8) {
            *reinterpret_cast<uint4*>(pm) = make_uint4(pack_bf16x2(mu[0], mu[1]), pack_bf16x2(mu[2], mu[3]),
                                                       pack_bf16x2(mu[4 % NO], mu[5 % NO]), pack_bf16x2(mu[6 % NO], mu[7 % NO]));
            *reinterpret_cast<uint4*>(pv) = make_uint4(pack_bf16x2(vr[0], vr[1]), pack_bf16x2(vr[2], vr[3]),
                                                       pack_bf16x2(vr[4 % NO], vr[5 % NO]), pack_bf16x2(vr[6 % NO], vr[7 % NO]));
          } else {
            *reinterpret_cast<uint2*>(pm) = make_uint2(pack_bf16x2(mu[0], mu[1]), pack_bf16x2(mu[2], mu[3]));
            *reinterpret_cast<uint2*>(pv) = make_uint2(pack_bf16x2(vr[0], vr[1]), pack_bf16x2(vr[2], vr[3]));
          }
          if (gl == 0 && tw == 0) {
            *reinterpret_cast<uint4*>(gi + tile_image_off(pl, 32, 34)) =
                make_uint4(pack_bf16x2(W / (float)a.V, 0.f), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(gi + tile_image_off(pl, 33, 34)) = make_uint4(0x3F803F80u, 0u, 0u, 0u);  // 1, 1: bias columns of geometry_fc
            a.nvalid[pl] = nval;
          }
        }
      }
      TS();  // 17: pool2 + outputs done
      tc_fence_before_sync();
    }
#undef TS
  }
  __syncthreads();
  if (warp == W_ISSUE) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 256);
  }
}

}  // namespace

// ---------------------------------------------------------------------------
// host: weight images in the twin column layouts
// ---------------------------------------------------------------------------
size_t view_twin3_bytes(int kind) { (void)kind; return (size_t)(512 * 1024); }

int view_twin3_build(dyn_net* n, const float* P, void* dst_dev, size_t dst_bytes, cudaStream_t st) {
  std::vector<uint8_t> img;
  std::vector<FusedChunk> tab;
  constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;
  // fold_bias: the layer's bias rides in the map's kBiasHi / kBiasLo columns
  auto add = [&](const LinearP& l, int N, int Npad, int Kpad, std::vector<int> map, float scale = 1.f,
                 bool fold_bias = false, float bias_scale = -1.f) {
    HostLayer L;
    L.W = P + l.w; L.N = N; L.Kw = l.in; L.Npad = Npad; L.Kpad = Kpad; L.colmap = std::move(map);
    L.scale = scale; L.bias_scale = bias_scale;
    if (fold_bias) L.bias = P + l.b;
    append_layer(L, img, tab, 0, 0, 9, true, kTwinStage);
  };
  auto add_plan = [&](const LinearP& l, int N, int Kpad, std::vector<int> map, float scale, bool fold_bias,
                      float bias_scale, int d_col, int a_kg0, const LayerPlan& plan) {
    HostLayer L;
    L.W = P + l.w; L.N = N; L.Kw = l.in; L.Npad = N; L.Kpad = Kpad; L.colmap = std::move(map);
    L.scale = scale; L.bias_scale = bias_scale;
    if (fold_bias) L.bias = P + l.b;
    append_layer_plan(L, img, tab, d_col, a_kg0, plan, kTwinStage);
  };
  // the back half of both nets (base_fc.2, vis_fc, vis_fc2): two sub-rounds per layer, accumulators
  // alternating between TMEM columns [128,256) and [0,128)
  auto add_back_half = [&](const LinearP& base2, const LinearP& vis0, const LinearP& vis2, const LinearP& vis2_0) {
    std::vector<int> m4 = identity_map(256, 272);
    m4[256] = kBiasHi; m4[257] = kBiasLo;
    // base_fc.2: the operand columns 128..255 are finished first (k-steps 8-15), then 0..127 and the bias step
    add_plan(base2, 128, 272, m4, 1.f, true, kLog2e, 128, 0, {{{8, 8}}, {{0, 8}, {16, 1}}});
    // vis_fc.0 on x (columns [0,128), true units; w1 and bias in the epilogue)
    add_plan(vis0, 128, 128, identity_map(128, 128), kLog2e, false, -1.f, 0, 0, {{{0, 4}}, {{4, 4}}});
    // vis_fc.2 rows 0..127 on h (columns [128,256) = k-groups 16..31, exp2 scale) + bias step at k-groups 32, 33
    std::vector<int> m6 = identity_map(128, 144);
    m6[128] = kBiasHi; m6[129] = kBiasLo;
    add_plan(vis2, 128, 144, m6, 1.f, true, kLog2e, 128, 16, {{{0, 4}}, {{4, 4}, {8, 1}}});
    // vis_fc2.0 on x (vis1 and bias in the epilogue)
    add_plan(vis2_0, 128, 128, identity_map(128, 128), kLog2e, false, -1.f, 0, 0, {{{0, 4}}, {{4, 4}}});
  };
  if (n->kind == DYN_NET_STATIC) {
    const StaticLayout& L = n->sl;
    // layer 1: component-major PE; twin 0 = comps 0..4 (+1 pad), twin 1 = comps 5..8, ray_diff, pad
    std::vector<int> m1(112, -1);
    auto comp_col = [](int ci, int j) {  // j: 0 = x, 1..5 = cos f_k, 6..10 = sin f_k
      if (ci < 3) return j == 0 ? ci : (j <= 5 ? 3 + 3 * (j - 1) + ci : 18 + 3 * (j - 6) + ci);
      const int d = ci - 3;
      return j == 0 ? 33 + d : (j <= 5 ? 39 + 6 * (j - 1) + d : 69 + 6 * (j - 6) + d);
    };
    for (int ci = 0; ci < 5; ++ci)
      for (int j = 0; j < 11; ++j) m1[11 * ci + j] = comp_col(ci, j);
    for (int ci = 5; ci < 9; ++ci)
      for (int j = 0; j < 11; ++j) m1[56 + 11 * (ci - 5) + j] = comp_col(ci, j);
    for (int i = 0; i < 4; ++i) m1[100 + i] = 99 + i;
    m1[104] = kBiasHi; m1[105] = kBiasLo;
    add(L.ray_dir0, 256, 256, 112, m1, kLog2e, true);               // ELU on the exp2 scale
    add(L.ray_dir2, kF, 48, 256, identity_map(256, 256), kLn2);     // consumes log2(e) * ELU
    // layer 3: per twin 5 groups of [mean8 | var8 | feat8]; concat channel c: mean c, var 70+c, feat 140+c
    std::vector<int> m3(256, -1);
    auto chan = [](int tw, int slot) {  // concat channel (0..69) of a twin's slot, -1 = pad
      if (tw == 0) return slot < 19 ? slot : (slot < 37 ? 35 + (slot - 19) : -1);
      return slot < 16 ? 19 + slot : (slot < 33 ? 53 + (slot - 16) : -1);
    };
    for (int tw = 0; tw < 2; ++tw)
      for (int s = 0; s < 40; ++s) {
        const int c = chan(tw, s);
        if (c < 0) continue;
        const int base = 128 * tw + 24 * (s / 8) + (s % 8);
        m3[base] = c; m3[base + 8] = 70 + c; m3[base + 16] = 140 + c;
      }
    m3[103] = kBiasHi; m3[111] = kBiasLo;  // twin 0, slot 39 (unused): mean / var columns of group 4
    // base_fc.0 (K = 256: twin 0 at [0,120), twin 1 at [128,248)): the k-steps over the first three pooled groups
    // of both twins (0-3 and 8-11) run while the last two groups are being pooled
    add_plan(L.base0, 256, 256, m3, kLog2e, true, -1.f, 0, 0, {{{0, 4}, {8, 4}}, {{4, 4}, {12, 4}}});
    add_back_half(L.base2, L.vis0, L.vis2, L.vis2_0);
  } else {
    const DynamicLayout& L = n->dl;
    // twin 0: channels 0..18 (3 groups, cols 0..71), twin 1: channels 19..34 (2 groups, cols 72..119)
    std::vector<int> m3(128, -1);
    for (int s = 0; s < 24; ++s)
      if (s < 19) { const int b = 24 * (s / 8) + (s % 8); m3[b] = s; m3[b + 8] = 35 + s; m3[b + 16] = 70 + s; }
    for (int s = 0; s < 16; ++s) {
      const int c = 19 + s, b = 72 + 24 * (s / 8) + (s % 8);
      m3[b] = c; m3[b + 8] = 35 + c; m3[b + 16] = 70 + c;
    }
    m3[55] = kBiasHi; m3[63] = kBiasLo;  // twin 0, slot 23 (unused): mean / var columns of group 2
    add(L.base0, 256, 256, 128, m3, kLog2e, true);
    add_back_half(L.base2, L.vis0, L.vis2, L.vis2_0);
  }
  const size_t img_bytes = (img.size() + 255) & ~(size_t)255;
  const size_t need = img_bytes + tab.size() * sizeof(FusedChunk);
  if (need > dst_bytes) return fail(DYN_E_INVALID, "twin images need %zu bytes, have %zu", need, dst_bytes);
  DYN_CUDA(cudaMemcpyAsync(dst_dev, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  DYN_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(dst_dev) + img_bytes, tab.data(),
                           tab.size() * sizeof(FusedChunk), cudaMemcpyHostToDevice, st));
  DYN_CUDA(cudaStreamSynchronize(st));
  n->twin3.img = dst_dev;
  n->twin3.tab = reinterpret_cast<const FusedChunk*>(reinterpret_cast<char*>(dst_dev) + img_bytes);
  n->twin3.nchunks = (int)tab.size();
  if (tab.size() > (size_t)kMaxChunks) return fail(DYN_E_INVALID, "chunk table too long (%zu)", tab.size());
  return DYN_OK;
}

int launch_view_twin3(const dyn_net* n, ViewFusedArgs& a, int V, cudaStream_t st) {
  if (n->twin3.img == nullptr) return fail(DYN_E_INVALID, "net has no twin-warp view images");
  a.wimg = n->twin3.img;
  a.chunks = n->twin3.tab;
  a.nchunks = n->twin3.nchunks;
  // one-time set-up (profiling knob DYN_ABLATE, SM count, dynamic shared-memory opt-in of every instantiation)
  static int ablate = -1, sms = 0;
  if (ablate < 0) {
    const char* e = getenv("DYN_ABLATE");
    int dev = 0;
    DYN_CUDA(cudaGetDevice(&dev));
    DYN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DYN_CUDA(cudaFuncSetAttribute(view_twin3_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTwinSmem));
    DYN_CUDA(cudaFuncSetAttribute(view_twin3_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTwinSmem));
    DYN_CUDA(cudaFuncSetAttribute(view_twin3_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTwinSmem));
    DYN_CUDA(cudaFuncSetAttribute(view_twin3_kernel<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTwinSmem));
    ablate = e ? atoi(e) : 0;
  }
  a.ablate = ablate;
  const int VP = V <= 8 ? 8 : 16;
  const long long n_iter = (a.P * VP + 127) / 128;
  const long long slots = 2LL * sms;
  const int grid = (int)(n_iter < slots ? n_iter : slots);
  if (grid == 0) return DYN_OK;
  const bool st_net = n->kind == DYN_NET_STATIC;
  ProfScope prof(st_net ? PROF_VIEW_ST : PROF_VIEW_DY, st);
  if (st_net) {
    if (VP == 8) view_twin3_kernel<8, true><<<grid, 320, kTwinSmem, st>>>(a);
    else view_twin3_kernel<16, true><<<grid, 320, kTwinSmem, st>>>(a);
  } else {
    if (VP == 8) view_twin3_kernel<8, false><<<grid, 320, kTwinSmem, st>>>(a);
    else view_twin3_kernel<16, false><<<grid, 320, kTwinSmem, st>>>(a);
  }
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // namespace dyn
