// Row-local fused tcgen05 chains of the aggregation networks in the twin-warp structure of the per-view
// kernel (view_twin3.cu): TWO independent CTAs per SM, each with ONE 128-row tile whose rows are served by
// TWO threads (warps w and w + 4 share the TMEM lane quadrant w & 3 and split every layer's output columns),
// plus the MMA issuer (warp 8) and the weight producer (warp 9).  16 row warps share an SM and the two CTAs
// desynchronise, which is what the latency-bound epilogues need (profiles/r02_chain_kernels.md).
//
//   rgbhead_twin_kernel : static per-view colour-blending head + masked softmax over views
//                         (mlp_network.py:508-526)
//   point1_twin_kernel  : geometry_fc -> (+ sinusoid) -> Q | K | V projections
//                         (mlp_network.py:283-286 / :496, :84-86)
//   point2_twin_kernel  : attention fc + residual + LayerNorm -> heads
//                         (mlp_network.py:99-102, :291-315 / :503-506, first rgb_fc layer)
//
// Hidden activations that only feed another MMA live on the exp2 scale (log2(e) * ELU: 3 instructions per
// activation, fused_engine.cuh: elu_log2) with their biases folded into the MMA wherever the operand has a
// free k-step.
#include "fused_engine.cuh"
#include "nets.cuh"

namespace dyn {

using namespace tc;
using namespace fe;

namespace {

constexpr int kTStage = 16384;
constexpr int kTRing = 2;
constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;

__device__ __forceinline__ void pair_sync_tw(int pair) {
  asm volatile("bar.sync %0, 64;" ::"r"(pair + 1) : "memory");
}

struct TwinCta {
  uint8_t* smem;
  uint8_t* ring;
  float* cst;
  uint32_t bar0, tmem_base;
};

// common prologue of the twin chains: chunk table, barriers, TMEM (256 columns); `a_bytes` = operand tile size
template <int kConstFloats>
__device__ __forceinline__ TwinCta twin_prologue(uint8_t* smem, int a_bytes, FusedChunk* s_tab,
                                                 const FusedChunk* chunks, int nchunks, int extra_bars) {
  TwinCta c;
  c.smem = smem;
  c.ring = smem + a_bytes;
  c.cst = reinterpret_cast<float*>(c.ring + kTRing * kTStage);
  uint64_t* bars = reinterpret_cast<uint64_t*>(c.cst + kConstFloats);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  c.bar0 = smem_u32(bars);
  stage_chunks(s_tab, chunks, nchunks);
  if (threadIdx.x == 0) {
    init_barriers(c.bar0, /*pp=*/false, /*arrivals=*/128, kTRing);
    for (int i = 0; i < extra_bars; ++i) mbar_init(c.bar0 + 8u * (12 + i), 1);
    mbar_fence_init();
  }
  if ((threadIdx.x >> 5) == 8) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  c.tmem_base = *tmem_slot;
  return c;
}
__device__ __forceinline__ void twin_teardown(const TwinCta& c) {
  __syncthreads();
  if ((threadIdx.x >> 5) == 8) {
    tc_fence_after_sync();
    tmem_dealloc(c.tmem_base, 256);
  }
}
__device__ __forceinline__ void t_ready(uint32_t bar0) {
  fence_proxy_async_smem();
  tc_fence_before_sync();
  mbar_arrive(bar_aready(bar0, 0, kTRing));
}
__device__ __forceinline__ void t_wait(uint32_t bar0, uint32_t& acc_cnt) {
  mbar_wait(bar_acc(bar0, 0, kTRing), acc_cnt & 1);
  ++acc_cnt;
  tc_fence_after_sync();
}

// ---------------------------------------------------------------------------
// static colour-blending head (rows = (point, view slot), VP slots per point)
// operand tile (36 k-groups): [x 128 | vis2, ray_diff(4), 0 x 11 | hidden 128 | 1, 1, 0 x 14]
// constants: [0,64) ln2 * w_rgb4   [64] b_rgb4   [128,384) partial logits [2][128]
// ---------------------------------------------------------------------------
constexpr int kRhATile = 36 * 2048;
constexpr int kRhConst = 384;
constexpr int kRhSmem = kRhATile + kTRing * kTStage + kRhConst * 4 + 256;

template <int VP>
__global__ void __launch_bounds__(320, 2) rgbhead_twin_kernel(const __grid_constant__ RgbHeadArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(16) FusedChunk s_tab[16];
  const TwinCta c = twin_prologue<kRhConst>(smem, kRhATile, s_tab, a.chunks, a.nchunks, 1);
  float* cst = c.cst;
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int i = tid; i < 64; i += blockDim.x) cst[i] = a.params[a.o_wrgb4 + i] * kLn2;
  if (tid == 0) cst[64] = a.params[a.o_brgb4];
  __syncthreads();
  const int n_iter = (int)((a.P * VP + 127) / 128);

  if (warp == 9) {
    if ((tid & 31) < a.producers)
      producer_loop<false, kTRing, kTStage>(s_tab, a.nchunks, a.wimg, n_iter, c.ring, c.bar0, tid & 31, a.producers);
  } else if (warp == 8) {
    issuer_loop<false, 1, kTRing, kTStage>(s_tab, a.nchunks, n_iter, smem, c.ring, c.bar0, c.tmem_base, kRhATile);
  } else {
    const int tw = tid >> 7, r = tid & 127;
    uint8_t* arow = smem + (r >> 3) * 128 + (r & 7) * 16;
    const uint32_t tacc = tmem_addr(c.tmem_base, (uint32_t)((warp & 3) * 32), 0u);
    const int v = r % VP;
    const int pair = warp & 3;
    float* xch = cst + 128;
    uint32_t acc_cnt = 0, x_cnt = 0;
    const uint32_t xbar = c.bar0 + 8u * 12;  // the x block of this iteration has landed
    const uint8_t* ximg = reinterpret_cast<const uint8_t*>(a.X);
    const uint32_t atile = smem_u32(smem);
    auto issue_x = [&](int it2) {
      mbar_arrive_expect_tx(xbar, 32768u);
      bulk_g2s(atile, ximg + (size_t)it2 * 32768u, 32768u, xbar);
    };
    if (tid == 0 && (int)blockIdx.x < n_iter) issue_x((int)blockIdx.x);
    if (tw == 0) {  // persistent bias columns of rgb_fc.2: k-groups 34, 35 = [1, 1, 0 ...]
      float o[8] = {1.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      store8(arow, 272, o);
      store8(arow, 280, z);
    }
    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      const long long pl = ((long long)it * 128 + r) / VP;
      const bool pt_ok = pl < a.P;
      const bool valid = pt_ok && v < a.V;
      const long long m = pl * a.V + v;
      // operand: the x block is the bf16 tile image spilled by the per-view kernel (one 32 KB bulk copy per
      // 128 rows, issued one iteration ahead); twin 0 appends [vis2, ray_diff] at columns 128..132
      if (tw == 0) {
        float t[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (valid) {
          const float4 rd = __ldg(reinterpret_cast<const float4*>(a.ray_diff) + m);
          t[0] = a.vis2[m]; t[1] = rd.x; t[2] = rd.y; t[3] = rd.z; t[4] = rd.w;
        }
        store8(arow, 128, t);
        float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        store8(arow, 136, z);
      }
      // per-point part of rgb_fc.0 (GW, bias included; fp32 tile layout written by point2): this twin's 64
      // columns are loaded BEFORE the waits (L2 latency hides behind the bulk copy / MMA)
      const int c0 = 64 * tw;
      const uint8_t* gw = reinterpret_cast<const uint8_t*>(a.GW) + tile_f32_off(pt_ok ? pl : 0, c0 >> 2);
      float4 g[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] = __ldg(reinterpret_cast<const float4*>(gw + i * 2048));
      mbar_wait(xbar, x_cnt & 1); ++x_cnt;
      t_ready(c.bar0);
      t_wait(c.bar0, acc_cnt);  // rgb_fc.0, per-view part (weights x log2 e): accumulator on the exp2 scale
      // the MMA has consumed columns [0,144): prefetch the next iteration's x block behind it
      if (tid == 0 && it + (int)gridDim.x < n_iter) issue_x(it + (int)gridDim.x);
      // read-out pipelined in 16-column halves; the GW values of half h + 2 are requested as soon as half h has
      // consumed its own (g[0..3] serve the even halves, g[4..7] the odd ones)
      tmem_pipe16<4>(tacc, [&](int h) { return c0 + 16 * h; }, [&](int h, float* v) {
        const int gb = (h & 1) * 4;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          v[4 * i] = elu_log2(fmaf(g[gb + i].x, kLog2e, v[4 * i]));
          v[4 * i + 1] = elu_log2(fmaf(g[gb + i].y, kLog2e, v[4 * i + 1]));
          v[4 * i + 2] = elu_log2(fmaf(g[gb + i].z, kLog2e, v[4 * i + 2]));
          v[4 * i + 3] = elu_log2(fmaf(g[gb + i].w, kLog2e, v[4 * i + 3]));
        }
        if (h < 2) {
#pragma unroll
          for (int i = 0; i < 4; ++i) g[gb + i] = __ldg(reinterpret_cast<const float4*>(gw + (8 + 4 * h + i) * 2048));
        }
        store8(arow, 144 + c0 + 16 * h, v);
        store8(arow, 144 + c0 + 16 * h + 8, v + 8);
      });
      t_ready(c.bar0);
      // masked-softmax inputs of this row (twin 0 blends): loaded before the wait
      float mk = 0.f, c3[3] = {0.f, 0.f, 0.f};
      if (tw == 0 && valid) {
        mk = a.mask_eff[m];
        c3[0] = a.rgb_in[m * 3]; c3[1] = a.rgb_in[m * 3 + 1]; c3[2] = a.rgb_in[m * 3 + 2];
      }
      t_wait(c.bar0, acc_cnt);  // rgb_fc.2 (64, bias folded, exp2 scale) -> rgb_fc.4 logit: this twin's 32 columns
      {
        float acc[32];
        tmem_ld32(tacc + 32 * tw, acc);
        tmem_wait_ld();
        float part = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) part = fmaf(elu_log2(acc[i]), cst[32 * tw + i], part);
        xch[tw * 128 + r] = part;
      }
      tc_fence_before_sync();
      pair_sync_tw(pair);
      if (tw == 0) {
        const float logit = cst[64] + xch[r] + xch[128 + r];
        // masked softmax over the views of the point, blend source colours (mlp_network.py:523-525)
        float l = valid ? (mk == 0.f ? -1e9f : logit) : -INFINITY;
        float mx = l;
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
        if (VP == 16) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
        const float e = valid ? __expf(l - mx) : 0.f;
        const float den = group_sum<VP>(e);
        const float w = e / den;
        float b0 = group_sum<VP>(c3[0] * w), b1 = group_sum<VP>(c3[1] * w), b2 = group_sum<VP>(c3[2] * w);
        if (pt_ok && v == 0) reinterpret_cast<float4*>(a.raw)[pl] = make_float4(b0, b1, b2, a.sigma[pl]);
      }
      // (the exchange slots are rewritten only after the next iteration's first MMA, which needs twin 0's
      //  arrival on a_ready, i.e. after twin 0 has read them)
    }
  }
  twin_teardown(c);
}

// NB blocks of 32 accumulator columns [col0 + 32 b, ..) -> ELU on the exp2 scale -> bf16 operand columns
// [dst0 + 32 b, ..); the TMEM read-out is software-pipelined in 16-column halves (fused_engine.cuh: tmem_pipe16)
template <int NB>
__device__ __forceinline__ void t_elu_log2_blocks(uint8_t* arow, uint32_t tacc, int col0, int dst0) {
  tmem_pipe16<2 * NB>(tacc, [&](int h) { return col0 + 16 * h; }, [&](int h, float* v) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = elu_log2(v[i]);
    store8(arow, dst0 + 16 * h, v);
    store8(arow, dst0 + 16 * h + 8, v + 8);
  });
}
// NB blocks of 32 accumulator columns -> bf16 tile image rows (16 k-groups: 4 per block starting at kgroup0),
// zeros for rows past the end
template <int NB>
__device__ __forceinline__ void t_store_image_blocks(uint32_t tacc, int col0, void* img, long long row, int kgroup0,
                                                     bool valid) {
  uint8_t* o = reinterpret_cast<uint8_t*>(img) + tile_image_off(row, kgroup0, 16);
  tmem_pipe16<2 * NB>(tacc, [&](int h) { return col0 + 16 * h; }, [&](int h, float* v) {
    if (!valid) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
      *reinterpret_cast<uint4*>(o + (2 * h + i) * 2048) =
          make_uint4(pack_bf16x2(v[8 * i], v[8 * i + 1]), pack_bf16x2(v[8 * i + 2], v[8 * i + 3]),
                     pack_bf16x2(v[8 * i + 4], v[8 * i + 5]), pack_bf16x2(v[8 * i + 6], v[8 * i + 7]));
  });
}

// ---------------------------------------------------------------------------
// per-point stage 1: G -> geometry_fc -> (+ posenc) -> g2, Q, K, V      (rows = points)
// operand tile = the G tile image (34 k-groups: mean 128 | var 128 | weight, 0 x 7 | 0 x 8 with 1, 1 at
// columns 264, 265: the per-view kernels write those ones, both geometry_fc biases ride on them)
// ---------------------------------------------------------------------------
constexpr int kP1ATile = 34 * 2048;
constexpr int kP1Const = 16;
constexpr int kP1Smem = kP1ATile + kTRing * kTStage + kP1Const * 4 + 256;

__global__ void __launch_bounds__(320, 2) point1_twin_kernel(const __grid_constant__ Point1Args a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(16) FusedChunk s_tab[32];
  const TwinCta c = twin_prologue<kP1Const>(smem, kP1ATile, s_tab, a.chunks, a.nchunks, 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int n_iter = (int)((a.P + 127) / 128);
  if (warp == 9) {
    if ((tid & 31) < a.producers)
      producer_loop<false, kTRing, kTStage>(s_tab, a.nchunks, a.wimg, n_iter, c.ring, c.bar0, tid & 31, a.producers);
  } else if (warp == 8) {
    issuer_loop<false, 1, kTRing, kTStage>(s_tab, a.nchunks, n_iter, smem, c.ring, c.bar0, c.tmem_base, kP1ATile);
  } else {
    const int tw = tid >> 7, r = tid & 127;
    uint8_t* arow = smem + (r >> 3) * 128 + (r & 7) * 16;
    const uint32_t tacc = tmem_addr(c.tmem_base, (uint32_t)((warp & 3) * 32), 0u);
    uint32_t acc_cnt = 0, g_cnt = 0;
    const uint32_t gbar = c.bar0 + 8u * 12;  // this iteration's G block has landed
    const uint8_t* gimg = reinterpret_cast<const uint8_t*>(a.G);
    const uint32_t atile = smem_u32(smem);
    auto issue_g = [&](int it2) {
      mbar_arrive_expect_tx(gbar, (uint32_t)kP1ATile);
      bulk_g2s(atile, gimg + (size_t)it2 * (size_t)kP1ATile, (uint32_t)kP1ATile, gbar);
    };
    if (tid == 0 && (int)blockIdx.x < n_iter) issue_g((int)blockIdx.x);
    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      const long long row = (long long)it * 128 + r;
      const bool valid = row < a.P;
      // operand: the pooled statistics arrive as a ready-made tile image (one 68 KB bulk copy per 128 points)
      mbar_wait(gbar, g_cnt & 1); ++g_cnt;
      t_ready(c.bar0);
      t_wait(c.bar0, acc_cnt);  // geometry_fc.0 (bias folded, exp2 scale): this twin's 128 of 256 columns
      t_elu_log2_blocks<4>(arow, tacc, 128 * tw, 128 * tw);
      t_ready(c.bar0);
      t_wait(c.bar0, acc_cnt);  // geometry_fc.2 (+ sinusoid for the dynamic net) -> g2: this twin's 64 columns
      {
        const int s_idx = valid ? (int)(row % a.S) : 0;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int cb = 64 * tw + 32 * half;
          float acc[32];
          tmem_ld32(tacc + cb, acc);
          float4 pe[8];
          if (a.posenc) {
#pragma unroll
            for (int i = 0; i < 8; ++i) pe[i] = __ldg(reinterpret_cast<const float4*>(a.posenc + s_idx * 128 + cb) + i);
          }
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = elu_from_log2(acc[i]);
          if (a.posenc) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              acc[4 * i] += pe[i].x; acc[4 * i + 1] += pe[i].y; acc[4 * i + 2] += pe[i].z; acc[4 * i + 3] += pe[i].w;
            }
          }
          if (valid) {  // residual stream, fp32 tile layout (fused_engine.cuh: tile_f32_off)
            uint8_t* o = reinterpret_cast<uint8_t*>(a.g2) + tile_f32_off(row, cb >> 2);
#pragma unroll
            for (int i = 0; i < 8; ++i)
              *reinterpret_cast<float4*>(o + i * 2048) = make_float4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) store8(arow, cb + 8 * g, acc + 8 * g);
        }
      }
      t_ready(c.bar0);
      t_wait(c.bar0, acc_cnt);  // [Wq ; Wk] (N = 256, no bias): twin 0 stores Q, twin 1 stores K (bf16 tile images)
      t_store_image_blocks<4>(tacc, 128 * tw, tw == 0 ? (void*)a.Q : (void*)a.K, row, 0, valid);
      tc_fence_before_sync();
      mbar_arrive(bar_aready(c.bar0, 0, kTRing));  // operand unchanged; the accumulators are free again
      t_wait(c.bar0, acc_cnt);                     // Wv
      if (tid == 0 && it + (int)gridDim.x < n_iter) issue_g(it + (int)gridDim.x);  // the operand tile is free
      t_store_image_blocks<2>(tacc, 64 * tw, a.V, row, 8 * tw, valid);
      tc_fence_before_sync();
    }
  }
  twin_teardown(c);
}

// ---------------------------------------------------------------------------
// per-point stage 2: fc(O) + g2 -> LayerNorm -> heads                    (rows = points)
// constants: [0,128) ln_w  [128,256) ln_b  [256,384) ln2 * w_outgeo2  [384,576) ln2 * w_rgb4 (3 x 64)
//            [576] b_outgeo2  [577..579] b_rgb4   exchange: [640, 640 + 6 x 256)
// ---------------------------------------------------------------------------
constexpr int kP2ATile = 34 * 2048;
constexpr int kP2X = 640;
constexpr int kP2Const = kP2X + 6 * 256;
constexpr int kP2Smem = kP2ATile + kTRing * kTStage + kP2Const * 4 + 256;

template <bool DYNAMIC>
__global__ void __launch_bounds__(320, 2) point2_twin_kernel(const __grid_constant__ Point2Args a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(16) FusedChunk s_tab[32];
  const TwinCta c = twin_prologue<kP2Const>(smem, kP2ATile, s_tab, a.chunks, a.nchunks, 1);
  float* cst = c.cst;
  const int tid = threadIdx.x, warp = tid >> 5;
  {
    const float* p = a.params;
    for (int i = tid; i < 128; i += blockDim.x) {
      cst[i] = p[a.o_lnw + i]; cst[128 + i] = p[a.o_lnb + i];
      cst[256 + i] = p[a.o_woutgeo2 + i] * kLn2;
    }
    if (DYNAMIC) {
      for (int i = tid; i < 192; i += blockDim.x) cst[384 + i] = p[a.o_wrgb4 + i] * kLn2;
      if (tid < 3) cst[577 + tid] = p[a.o_brgb4 + tid];
    }
    if (tid == 0) cst[576] = p[a.o_boutgeo2];
  }
  __syncthreads();
  const int n_iter = (int)((a.P + 127) / 128);
  if (warp == 9) {
    if ((tid & 31) < a.producers)
      producer_loop<false, kTRing, kTStage>(s_tab, a.nchunks, a.wimg, n_iter, c.ring, c.bar0, tid & 31, a.producers);
  } else if (warp == 8) {
    issuer_loop<false, 1, kTRing, kTStage>(s_tab, a.nchunks, n_iter, smem, c.ring, c.bar0, c.tmem_base, kP2ATile);
  } else {
    const int tw = tid >> 7, r = tid & 127;
    uint8_t* arow = smem + (r >> 3) * 128 + (r & 7) * 16;
    const uint32_t tacc = tmem_addr(c.tmem_base, (uint32_t)((warp & 3) * 32), 0u);
    const int pair = warp & 3;
    float* x_sum = cst + kP2X;          // [2][128] LayerNorm partial sums
    float* x_sq = cst + kP2X + 256;     // [2][128]
    float* x_sig = cst + kP2X + 512;    // [2][128] density-head partial dot products
    float* x_rgb = cst + kP2X + 768;    // [3][2][128] colour-head partial dot products (dynamic)
    uint32_t acc_cnt = 0, o_cnt = 0;
    const uint32_t obar = c.bar0 + 8u * 12;
    const uint8_t* oimg = reinterpret_cast<const uint8_t*>(a.O);
    const uint32_t atile = smem_u32(smem);
    auto issue_o = [&](int it2) {
      mbar_arrive_expect_tx(obar, 32768u);
      bulk_g2s(atile, oimg + (size_t)it2 * 32768u, 32768u, obar);
    };
    if (tid == 0 && (int)blockIdx.x < n_iter) issue_o((int)blockIdx.x);
    if (tw == 0) {
      // persistent bias columns: static [out_geometry_fc.0 | rgb_fc.0] round reads k-groups 16, 17;
      // dynamic ref_pts_fc.2 reads k-groups 32, 33
      float o[8] = {1.f, 1.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      store8(arow, DYNAMIC ? 256 : 128, o);
      store8(arow, DYNAMIC ? 264 : 136, z);
    }
    const int c0 = 64 * tw;
    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      const long long row = (long long)it * 128 + r;
      const bool valid = row < a.P;
      // residual (fp32 tile layout), this twin's 64 columns: loaded before the waits
      const uint8_t* res = reinterpret_cast<const uint8_t*>(a.g2) + tile_f32_off(valid ? row : 0, c0 >> 2);
      float4 rs[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) rs[i] = valid ? __ldg(reinterpret_cast<const float4*>(res + i * 2048)) : make_float4(0.f, 0.f, 0.f, 0.f);
      // operand: attention output O, a bf16 tile image: one 32 KB bulk copy per 128 points
      mbar_wait(obar, o_cnt & 1); ++o_cnt;
      t_ready(c.bar0);
      t_wait(c.bar0, acc_cnt);  // fc (no bias) + residual; LayerNorm (eps 1e-6) statistics via TMEM scratch
      {
        float sum = 0.f, sq = 0.f;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int cb = c0 + 32 * half;
          float acc[32];
          tmem_ld32(tacc + cb, acc);
          if (half == 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              rs[i] = valid ? __ldg(reinterpret_cast<const float4*>(res + (8 + i) * 2048)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            acc[4 * i] += rs[i].x; acc[4 * i + 1] += rs[i].y; acc[4 * i + 2] += rs[i].z; acc[4 * i + 3] += rs[i].w;
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) { sum += acc[i]; sq = fmaf(acc[i], acc[i], sq); }
          tmem_st32(tacc + 128 + cb, acc);
        }
        x_sum[tw * 128 + r] = sum;
        x_sq[tw * 128 + r] = sq;
        tmem_wait_st();
        pair_sync_tw(pair);
        sum = x_sum[r] + x_sum[128 + r];
        sq = x_sq[r] + x_sq[128 + r];
        const float mean = sum * (1.f / 128.f);
        const float var = fmaxf(sq * (1.f / 128.f) - mean * mean, 0.f);
        const float rstd = rsqrtf(var + 1e-6f);
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int cb = c0 + 32 * half;
          float y[32];
          tmem_ld32(tacc + 128 + cb, y);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) y[i] = (y[i] - mean) * rstd * cst[cb + i] + cst[128 + cb + i];
#pragma unroll
          for (int g = 0; g < 4; ++g) store8(arow, cb + 8 * g, y + 8 * g);
        }
      }
      if (DYNAMIC) {
        if (tw == 0) {
          // append PE(pts) (33) at columns 128..160, the bias ones of ref_pts_fc.0 at 161, 162, zeros to 175
          float p3[3] = {0.f, 0.f, 0.f};
          if (valid) { p3[0] = a.pts[row * 3]; p3[1] = a.pts[row * 3 + 1]; p3[2] = a.pts[row * 3 + 2]; }
          float pe[48];
          pe_pow2<3, 5>(p3, pe);
          pe[33] = 1.f; pe[34] = 1.f;
#pragma unroll
          for (int i = 35; i < 48; ++i) pe[i] = 0.f;
#pragma unroll
          for (int g = 0; g < 6; ++g) store8(arow, 128 + 8 * g, pe + 8 * g);
        }
        t_ready(c.bar0);
        t_wait(c.bar0, acc_cnt);  // ref_pts_fc.0 (K = 176, bias folded, exp2 scale): this twin's 128 of 256 columns
        t_elu_log2_blocks<4>(arow, tacc, 128 * tw, 128 * tw);
        t_ready(c.bar0);
        t_wait(c.bar0, acc_cnt);  // ref_pts_fc.2 (K = 256 + bias step) -> g4 on the exp2 scale: 64 columns
        t_elu_log2_blocks<2>(arow, tacc, c0, c0);
        if (tw == 1) {
          // append PE(dir) (27) at columns 128..154, the bias ones of the next two rounds at 155, 156
          const long long ray = valid ? row / a.S : 0;
          float d3[3] = {a.ray_dir[ray * 3], a.ray_dir[ray * 3 + 1], a.ray_dir[ray * 3 + 2]};
          float pe2[32];
          pe_pow2<3, 4>(d3, pe2);
          pe2[27] = 1.f; pe2[28] = 1.f;
#pragma unroll
          for (int i = 29; i < 32; ++i) pe2[i] = 0.f;
#pragma unroll
          for (int g = 0; g < 4; ++g) store8(arow, 128 + 8 * g, pe2 + 8 * g);
        }
      }
      t_ready(c.bar0);
      // round: out_geometry_fc.0 -> accumulator columns [0,128) (exp2 scale), rgb_fc.0 (dynamic, exp2 scale) /
      // rgb_fc.0[:, :128] (static, true scale, bias included = GW) -> [128,256)
      const float nv = valid ? a.nvalid[row] : 0.f;
      t_wait(c.bar0, acc_cnt);
      if (!DYNAMIC && tid == 0 && it + (int)gridDim.x < n_iter) issue_o(it + (int)gridDim.x);  // last MMA round is done
      {
        float part = 0.f;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int cb = c0 + 32 * half;
          float acc[32];
          tmem_ld32(tacc + cb, acc);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) part = fmaf(elu_log2(acc[i]), cst[256 + cb + i], part);
        }
        x_sig[tw * 128 + r] = part;
      }
      if (DYNAMIC) {
        t_elu_log2_blocks<2>(arow, tacc, 128 + c0, c0);  // ELU(rgb_fc.0) -> operand columns [0,128)
        t_ready(c.bar0);
        t_wait(c.bar0, acc_cnt);  // rgb_fc.2 (64, bias folded, exp2 scale) -> rgb_fc.4 (3) as dot products: 32 columns
        if (tid == 0 && it + (int)gridDim.x < n_iter) issue_o(it + (int)gridDim.x);
        {
          float acc[32];
          tmem_ld32(tacc + 32 * tw, acc);
          tmem_wait_ld();
          float q0 = 0.f, q1 = 0.f, q2 = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float h = elu_log2(acc[i]);
            q0 = fmaf(h, cst[384 + 32 * tw + i], q0);
            q1 = fmaf(h, cst[384 + 64 + 32 * tw + i], q1);
            q2 = fmaf(h, cst[384 + 128 + 32 * tw + i], q2);
          }
          x_rgb[tw * 128 + r] = q0;
          x_rgb[256 + tw * 128 + r] = q1;
          x_rgb[512 + tw * 128 + r] = q2;
        }
        tc_fence_before_sync();
        pair_sync_tw(pair);
        if (tw == 0 && valid) {
          const float sigma = cst[576] + x_sig[r] + x_sig[128 + r];
          const float r0 = cst[577] + x_rgb[r] + x_rgb[128 + r];
          const float r1 = cst[578] + x_rgb[256 + r] + x_rgb[256 + 128 + r];
          const float r2 = cst[579] + x_rgb[512 + r] + x_rgb[512 + 128 + r];
          const bool none = nv < 1.f;  // mlp_network.py:297-299, :314
          reinterpret_cast<float4*>(a.raw)[row] =
              make_float4(none ? 0.f : sigmoid_fast(r0), none ? 0.f : sigmoid_fast(r1),
                          none ? 0.f : sigmoid_fast(r2), none ? -1e9f : sigma - a.shift);
        }
      } else {
        // static: per-point part of the blending head, GW = rgb_fc.0[:, :128] g + b (bias folded), fp32 tile layout
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int cb = c0 + 32 * half;
          float acc[32];
          tmem_ld32(tacc + 128 + cb, acc);
          tmem_wait_ld();
          if (valid) {
            uint8_t* o = reinterpret_cast<uint8_t*>(a.GW) + tile_f32_off(row, cb >> 2);
#pragma unroll
            for (int i = 0; i < 8; ++i)
              *reinterpret_cast<float4*>(o + i * 2048) = make_float4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
          }
        }
        tc_fence_before_sync();
        pair_sync_tw(pair);
        if (tw == 0 && valid) a.sigma[row] = nv < 1.f ? -1e9f : cst[576] + x_sig[r] + x_sig[128 + r];
      }
      // (the exchange slots are rewritten only after the next iteration's first MMA round, which needs both
      //  twins' arrivals, i.e. after twin 0 has read them)
    }
  }
  twin_teardown(c);
}

template <class K, class A>
int launch_twin(K kernel, const A& args, long long rows, int smem_bytes, cudaStream_t st) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    DYN_CUDA(cudaGetDevice(&dev));
    DYN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const long long n_iter = (rows + 127) / 128;
  const int grid = (int)(n_iter < 2LL * sms ? n_iter : 2LL * sms);
  if (grid == 0) return DYN_OK;
  kernel<<<grid, 320, smem_bytes, st>>>(args);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // namespace

// ---------------------------------------------------------------------------
// host: weight images of the twin chains
// ---------------------------------------------------------------------------
size_t twin_chain_bytes(int kind) { return kind == DYN_NET_MOTION ? 0 : (size_t)(768 * 1024); }

static int upload_twin(std::vector<uint8_t>& img, std::vector<FusedChunk>& tab, char*& cursor, size_t& left,
                       ChainImage* out, cudaStream_t st) {
  const size_t img_bytes = (img.size() + 255) & ~(size_t)255;
  const size_t need = img_bytes + ((tab.size() * sizeof(FusedChunk) + 255) & ~(size_t)255);
  if (need > left) return fail(DYN_E_INVALID, "twin chain images need %zu bytes, have %zu", need, left);
  DYN_CUDA(cudaMemcpyAsync(cursor, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  DYN_CUDA(cudaMemcpyAsync(cursor + img_bytes, tab.data(), tab.size() * sizeof(FusedChunk), cudaMemcpyHostToDevice, st));
  DYN_CUDA(cudaStreamSynchronize(st));
  out->img = cursor;
  out->tab = reinterpret_cast<const FusedChunk*>(cursor + img_bytes);
  out->nchunks = (int)tab.size();
  cursor += need;
  left -= need;
  img.clear();
  tab.clear();
  return DYN_OK;
}

int twin_chain_build(dyn_net* n, const float* P, void* dst_dev, size_t dst_bytes, cudaStream_t st) {
  if (n->kind == DYN_NET_MOTION) return DYN_OK;
  std::vector<uint8_t> img;
  std::vector<FusedChunk> tab;
  char* cur = reinterpret_cast<char*>(dst_dev);
  size_t left = dst_bytes;
  auto add = [&](const LinearP& l, int N, int Npad, int Kpad, std::vector<int> map, float scale, bool fold_bias,
                 float bias_scale, int a_kg0) {
    HostLayer L;
    L.W = P + l.w; L.N = N; L.Kw = l.in; L.Npad = Npad; L.Kpad = Kpad; L.colmap = std::move(map);
    L.scale = scale; L.bias_scale = bias_scale;
    if (fold_bias) L.bias = P + l.b;
    append_layer(L, img, tab, 0, a_kg0, 9, true, kTStage);
  };
  {
    const bool dynamic = n->kind == DYN_NET_DYNAMIC;
    const LinearP &geo0 = dynamic ? n->dl.geo0 : n->sl.geo0, &geo2 = dynamic ? n->dl.geo2 : n->sl.geo2;
    const LinearP &wq = dynamic ? n->dl.wq : n->sl.wq, &wk = dynamic ? n->dl.wk : n->sl.wk;
    const LinearP &wv = dynamic ? n->dl.wv : n->sl.wv, &fc = dynamic ? n->dl.fc : n->sl.fc;
    const LinearP &og0 = dynamic ? n->dl.outgeo0 : n->sl.outgeo0;
    // K columns followed by pad and the folded bias at operand columns hi, hi + 1
    auto with_bias = [](int K, int Kpad, int hi) {
      std::vector<int> m = identity_map(K, Kpad);
      m[hi] = kBiasHi; m[hi + 1] = kBiasLo;
      return m;
    };
    // ---- point stage 1: geometry_fc.0 (K = 272: G image, ones at 264, 265), geometry_fc.2 (K = 256 + the
    //      same two columns), [Wq ; Wk] as one N = 256 layer, Wv
    add(geo0, 256, 256, 272, with_bias(257, 272, 264), kLog2e, true, -1.f, 0);
    add(geo2, 128, 128, 272, with_bias(256, 272, 264), 1.f, true, kLog2e, 0);
    {
      std::vector<float> qk(256 * 128);
      memcpy(qk.data(), P + wq.w, 128 * 128 * sizeof(float));
      memcpy(qk.data() + 128 * 128, P + wk.w, 128 * 128 * sizeof(float));
      HostLayer L;
      L.W = qk.data(); L.N = 256; L.Kw = 128; L.Npad = 256; L.Kpad = 128; L.colmap = identity_map(128, 128);
      append_layer(L, img, tab, 0, 0, 9, true, kTStage);
    }
    add(wv, 128, 128, 128, identity_map(128, 128), 1.f, false, -1.f, 0);
    int rc = upload_twin(img, tab, cur, left, &n->chain_tw[0], st);
    if (rc) return rc;
    // ---- point stage 2
    add(fc, 128, 128, 128, identity_map(128, 128), 1.f, false, -1.f, 0);
    auto add2 = [&](const LinearP& l, int N, int Kpad, std::vector<int> map, float scale, float bias_scale,
                    std::vector<float> colscale, int d_col, int first_flags, bool last) {
      HostLayer L;
      L.W = P + l.w; L.N = N; L.Kw = l.in; L.Npad = N; L.Kpad = Kpad; L.colmap = std::move(map);
      L.scale = scale; L.bias_scale = bias_scale; L.bias = P + l.b; L.colscale = std::move(colscale);
      append_layer(L, img, tab, d_col, 0, first_flags, last, kTStage);
    };
    if (dynamic) {
      // ref_pts_fc.0 on [y 128 | PE(pts) 33 | 1 1 | 0]; ref_pts_fc.2 consumes the exp2-scale hidden layer
      add(n->dl.refpts0, 256, 256, 176, with_bias(161, 176, 161), kLog2e, true, -1.f, 0);
      add(n->dl.refpts2, 128, 128, 272, with_bias(256, 272, 256), 1.f, true, kLog2e, 0);
      // operand [g4 (exp2 scale) 128 | PE(dir) 27 | 1 1 | 0]: g4 columns x ln2, both outputs on the exp2 scale
      std::vector<float> cs(160, 1.f);
      for (int i = 0; i < 128; ++i) cs[i] = kLn2;
      add2(og0, 128, 160, with_bias(128, 160, 155), kLog2e, kLog2e, cs, 0, 9, false);
      add2(n->dl.rgb0, 128, 160, with_bias(155, 160, 155), kLog2e, kLog2e, cs, 128, 8, true);
      // rgb_fc.2 on [hidden (exp2 scale) 128 | (PE(dir): zero weights) | 1 1]
      add2(n->dl.rgb2, 64, 160, with_bias(128, 160, 155), 1.f, kLog2e, {}, 0, 9, true);
    } else {
      // operand [y 128 | 1 1 | 0]: out_geometry_fc.0 on the exp2 scale, rgb_fc.0[:, :128] + b in true units (= GW)
      add2(og0, 128, 144, with_bias(128, 144, 128), kLog2e, kLog2e, {}, 0, 9, false);
      add2(n->sl.rgb0, 128, 144, with_bias(128, 144, 128), 1.f, 1.f, {}, 128, 8, true);
    }
    rc = upload_twin(img, tab, cur, left, &n->chain_tw[1], st);
    if (rc) return rc;
  }
  if (n->kind == DYN_NET_STATIC) {
    // blending head: operand [x 128 | vis2, ray_diff 4 | pad] <-> rgb_fc.0 columns 128..260 (the per-point
    // columns 0..127 and the bias arrive as GW); hidden layer at columns [144,272), its bias at 272, 273
    std::vector<int> m(144, -1);
    for (int i = 0; i < 133; ++i) m[i] = 128 + i;
    add(n->sl.rgb0, 128, 128, 144, m, kLog2e, false, -1.f, 0);
    std::vector<int> m2 = identity_map(128, 144);
    m2[128] = kBiasHi; m2[129] = kBiasLo;
    add(n->sl.rgb2, 64, 64, 144, m2, 1.f, true, kLog2e, 18);
    int rc = upload_twin(img, tab, cur, left, &n->chain_tw[2], st);
    if (rc) return rc;
  }
  return DYN_OK;
}

int launch_point1_twin(const dyn_net* n, Point1Args& a, cudaStream_t st) {
  if (!n->chain_tw[0].img) return fail(DYN_E_INVALID, "net has no twin point-stage images");
  a.wimg = n->chain_tw[0].img; a.chunks = n->chain_tw[0].tab; a.nchunks = n->chain_tw[0].nchunks;
  a.params = n->params;
  a.producers = producer_lanes();
  static bool prepared = false;
  if (!prepared) {
    DYN_CUDA(cudaFuncSetAttribute(point1_twin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kP1Smem));
    prepared = true;
  }
  ProfScope prof(PROF_POINT1, st);
  return launch_twin(point1_twin_kernel, a, a.P, kP1Smem, st);
}

int launch_point2_twin(const dyn_net* n, Point2Args& a, cudaStream_t st) {
  if (!n->chain_tw[1].img) return fail(DYN_E_INVALID, "net has no twin point-stage images");
  const bool dynamic = n->kind == DYN_NET_DYNAMIC;
  a.wimg = n->chain_tw[1].img; a.chunks = n->chain_tw[1].tab; a.nchunks = n->chain_tw[1].nchunks;
  a.params = n->params;
  a.producers = producer_lanes();
  a.shift = n->shift;
  static bool prepared = false;
  if (!prepared) {
    DYN_CUDA(cudaFuncSetAttribute(point2_twin_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kP2Smem));
    DYN_CUDA(cudaFuncSetAttribute(point2_twin_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kP2Smem));
    prepared = true;
  }
  ProfScope prof(PROF_POINT2, st);
  if (dynamic) {
    const DynamicLayout& L = n->dl;
    a.o_lnw = L.ln_w; a.o_lnb = L.ln_b; a.o_woutgeo2 = L.outgeo2.w; a.o_boutgeo2 = L.outgeo2.b;
    a.o_wrgb4 = L.rgb4.w; a.o_brgb4 = L.rgb4.b;
    return launch_twin(point2_twin_kernel<true>, a, a.P, kP2Smem, st);
  }
  const StaticLayout& L = n->sl;
  a.o_lnw = L.ln_w; a.o_lnb = L.ln_b; a.o_woutgeo2 = L.outgeo2.w; a.o_boutgeo2 = L.outgeo2.b;
  a.o_wrgb4 = 0; a.o_brgb4 = 0;
  return launch_twin(point2_twin_kernel<false>, a, a.P, kP2Smem, st);
}

int launch_rgbhead_twin(const dyn_net* n, RgbHeadArgs& a, cudaStream_t st) {
  if (!n->chain_tw[2].img) return fail(DYN_E_INVALID, "static net has no twin blending-head images");
  a.wimg = n->chain_tw[2].img; a.chunks = n->chain_tw[2].tab; a.nchunks = n->chain_tw[2].nchunks;
  a.params = n->params;
  a.producers = producer_lanes();
  a.o_brgb2 = n->sl.rgb2.b; a.o_wrgb4 = n->sl.rgb4.w; a.o_brgb4 = n->sl.rgb4.b;
  static bool prepared = false;
  if (!prepared) {
    DYN_CUDA(cudaFuncSetAttribute(rgbhead_twin_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRhSmem));
    DYN_CUDA(cudaFuncSetAttribute(rgbhead_twin_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRhSmem));
    prepared = true;
  }
  ProfScope prof(PROF_RGBHEAD, st);
  if (a.V <= 8) return launch_twin(rgbhead_twin_kernel<8>, a, a.P * 8, kRhSmem, st);
  return launch_twin(rgbhead_twin_kernel<16>, a, a.P * 16, kRhSmem, st);
}

}  // namespace dyn
