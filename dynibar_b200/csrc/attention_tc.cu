// Ray-transformer attention on tcgen05 (a11: ibrnet/mlp_network.py:13-31, :84-98).
//
// One CTA = one 128-row tile = 128/S whole rays (S | 128).  Q, K, V arrive as bf16 tile
// images (fused_engine.cuh; written by point1_twin_kernel) and are landed in shared memory
// by bulk copies (K, V: 32 KB each per tile; Q: one 8 KB head slice at a time);
// per head h:  logits = Q_h K_h^T  (UMMA 128x128x32, fp32 in TMEM columns [0,128))
//              softmax over the keys of the row's own ray, in registers
//              (query rows with <= 1 valid view attend uniformly: the reference
//               masks QUERY rows, mlp_network.py:23-24, :91-94)
//              O_h = P V_h        (UMMA 128x32x128; P is written back to smem as the
//               A operand, V_h is read in place as an MN-major B operand)
// O (fp32, TMEM columns [128,256)) is written to global at the end, again as a bf16 tile image.
#include "nets.cuh"
#include "tc.cuh"
#include <cstdlib>
#include <cstring>

namespace dyn {

using namespace tc;

namespace {

constexpr int kTile = 128 * 128 * 2;  // one bf16 [128 x 128] canonical tile: 32 KB
constexpr int kQSlice = 128 * 32 * 2;  // Q_h: [128 x 32] = 8 KB
// K, V, P tiles + Q_h slice + barriers/inv: 104 KB + 2.3 KB -> two CTAs per SM
// + barriers (256 B) + per-row partial softmax sums [2 twins][128][4 heads] + partial maxima [2][128]
constexpr int kSmemAttn = 3 * kTile + kQSlice + 256 + 2 * 128 * 4 * 4 + 2 * 128 * 4;

// idesc with B in MN-major layout (bit 16)
__host__ __device__ constexpr uint32_t idesc_bf16_f32_bmn(int M, int N) {
  return idesc_bf16_f32(M, N) | (1u << 16);
}

// TW: two threads per row in twin warps w, w+4 (same TMEM lane quadrant): each twin owns half of the
// row's keys in the softmax and half of every head's output dims (needs S % 64 == 0 so that a twin's
// key range is whole 32-column TMEM blocks).  16 row warps per SM instead of 8.
template <bool TW>
__global__ void __launch_bounds__(TW ? 256 : 128, 2)
attention_tc_kernel(const __nv_bfloat16* __restrict__ Q, const __nv_bfloat16* __restrict__ K,
                    const __nv_bfloat16* __restrict__ V, const float* __restrict__ nvalid, long long P, int S,
                    __nv_bfloat16* __restrict__ O) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* kt = smem;
  uint8_t* vt = smem + kTile;
  uint8_t* pt = smem + 2 * kTile;
  uint8_t* qt = smem + 3 * kTile;  // Q_h slice [128 x 32]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 3 * kTile + kQSlice);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar_s = smem_u32(bars), bar_o = smem_u32(bars + 1);
  const uint32_t bar_kv = smem_u32(bars + 2), bar_q = smem_u32(bars + 3);
  if (tid == 0) {
    mbar_init(bar_s, 1); mbar_init(bar_o, 1); mbar_init(bar_kv, 1); mbar_init(bar_q, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tacc = tmem_addr(tmem_base, (uint32_t)((warp & 3) * 32), 0);

  const int r = tid & 127, tw = tid >> 7;
  const int rw = warp & 3;  // row warp: rows 32 rw .. 32 rw + 31
  const size_t roff = (size_t)(r >> 3) * 128 + (r & 7) * 16;
  const int ray_lo = (r / S) * S;  // first key row (inside the tile) of this row's ray
  // this THREAD's keys [k_lo, k_hi) and the key range touched by ANY row of this warp (tcgen05.ld is
  // warp-collective: the column blocks a warp skips must be the same for all its lanes)
  const int k_lo = TW ? ray_lo + tw * (S >> 1) : ray_lo;
  const int k_hi = TW ? k_lo + (S >> 1) : ray_lo + S;
  const int warp_lo = TW ? k_lo : ((rw * 32) / S) * S;
  const int warp_hi = TW ? k_hi : ((rw * 32 + 31) / S + 1) * S;
  float* den_part = reinterpret_cast<float*>(bars + 8);        // [2][128][4]
  float* max_part = den_part + 2 * 128 * 4;                    // [2][128]
  const float scale = 0.17677669529663687f;  // 1 / sqrt(32)
  uint32_t ph_s = 0, ph_o = 0, ph_kv = 0, ph_q = 0;
  const uint8_t* qimg = reinterpret_cast<const uint8_t*>(Q);
  const uint8_t* kimg = reinterpret_cast<const uint8_t*>(K);
  const uint8_t* vimg = reinterpret_cast<const uint8_t*>(V);

  // thread 0 issues every bulk copy; the MMAs are issued by an elected lane of warp 0 with the
  // whole warp converged (descriptors then stay in uniform registers)
  auto issue_qk = [&](int h) {  // all lanes of warp 0: logits_h = Q_h K_h^T (waits for the Q_h slice)
    mbar_wait(bar_q, ph_q & 1); ++ph_q;
    tc_fence_after_sync();
    if (elect_one()) {
      const uint32_t idesc = idesc_bf16_f32(128, 128);
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        mma_bf16_ss(tmem_base, smem_desc(smem_u32(qt) + (2 * ks) * 2048u, 2048u, 128u),
                    smem_desc(smem_u32(kt) + (4 * h + 2 * ks) * 2048u, 2048u, 128u), idesc, ks ? 1u : 0u);
      mma_commit(bar_s);
    }
    __syncwarp();
  };
  auto load_q = [&](long long tile, int h) {  // head slice: k-groups 4h..4h+3 are contiguous in the image
    mbar_arrive_expect_tx(bar_q, (uint32_t)kQSlice);
    bulk_g2s(smem_u32(qt), qimg + (size_t)tile * kTile + (size_t)h * kQSlice, (uint32_t)kQSlice, bar_q);
  };

  const long long n_tiles = (P + 127) / 128;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row = tile * 128 + r;
    const bool ok = row < P;
    if (tid == 0) {
      mbar_arrive_expect_tx(bar_kv, 2u * kTile);
      bulk_g2s(smem_u32(kt), kimg + (size_t)tile * kTile, (uint32_t)kTile, bar_kv);
      bulk_g2s(smem_u32(vt), vimg + (size_t)tile * kTile, (uint32_t)kTile, bar_kv);
      load_q(tile, 0);
    }
    const bool q_valid = ok && nvalid[row] > 1.f;
    mbar_wait(bar_kv, ph_kv & 1); ++ph_kv;
    if (warp == 0) issue_qk(0);
    for (int h = 0; h < 4; ++h) {
      mbar_wait(bar_s, ph_s & 1);
      ++ph_s;
      tc_fence_after_sync();
      if (tid == 0 && h < 3) load_q(tile, h + 1);  // Q_h has been consumed
      // ---- softmax over this row's ray (keys [ray_lo, ray_lo + S)) ----
      float mx = -INFINITY;
#pragma unroll 1
      for (int cb = 0; cb < 128; cb += 32) {
        if (cb + 32 <= warp_lo || cb >= warp_hi) continue;
        float l[32];
        tmem_ld32(tacc + cb, l);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int key = cb + i;
          if (key >= k_lo && key < k_hi) mx = fmaxf(mx, q_valid ? l[i] * scale : 0.f);
        }
      }
      if (TW) {  // combine the twins' maxima
        max_part[tw * 128 + r] = mx;
        asm volatile("bar.sync %0, 64;" ::"r"(1 + rw) : "memory");
        mx = fmaxf(mx, max_part[(tw ^ 1) * 128 + r]);
      }
      float den = 0.f;
      // previous head's P V must be done before P is overwritten
      if (h > 0) { mbar_wait(bar_o, ph_o & 1); ++ph_o; tc_fence_after_sync(); }
#pragma unroll 1
      for (int cb = 0; cb < 128; cb += 32) {
        float p[32];
        const bool any = !(cb + 32 <= warp_lo || cb >= warp_hi);
        // twins: a block outside the warp's keys belongs to the other twin or to another ray; the
        // latter (P must be zero there) are split between the twins by block parity
        if (TW && !any && ((cb + 32 <= ray_lo || cb >= ray_lo + S) ? ((cb >> 5) & 1) != tw : true)) continue;
        if (any) {
          tmem_ld32(tacc + cb, p);
          tmem_wait_ld();
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int key = cb + i;
          float e = 0.f;
          if (any && key >= k_lo && key < k_hi) e = q_valid ? __expf(p[i] * scale - mx) : 1.f;
          p[i] = e;
          den += e;
        }
        // unnormalised probabilities -> bf16 A operand (normalisation folded into the output)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 q;
          q.x = pack_bf16x2(p[8 * g], p[8 * g + 1]); q.y = pack_bf16x2(p[8 * g + 2], p[8 * g + 3]);
          q.z = pack_bf16x2(p[8 * g + 4], p[8 * g + 5]); q.w = pack_bf16x2(p[8 * g + 6], p[8 * g + 7]);
          *reinterpret_cast<uint4*>(pt + roff + ((cb >> 3) + g) * 2048) = q;
        }
      }
      den_part[(tw * 128 + r) * 4 + h] = den;  // 1 / sum applied when O is written out
      fence_proxy_async_smem();
      tc_fence_before_sync();
      __syncthreads();  // P complete; every thread is done reading logits_h
      if (warp == 0) {
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t idesc = idesc_bf16_f32_bmn(128, 32);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            mma_bf16_ss(tmem_base + 128 + 32 * h, smem_desc(smem_u32(pt) + ks * 4096u, 2048u, 128u),
                        // V_h as MN-major B: n = d in [32h, 32h+32) -> n-groups at stride 2048 (SBO),
                        // k = key -> k-groups at stride 128 (LBO); this k-step covers keys [16ks, 16ks+16)
                        smem_desc(smem_u32(vt) + (4 * h) * 2048u + ks * 256u, 128u, 2048u), idesc,
                        ks ? 1u : 0u);
          mma_commit(bar_o);
        }
        __syncwarp();
        if (h < 3) issue_qk(h + 1);  // queued behind P V_h; overlaps the next softmax's wait
      }
    }
    mbar_wait(bar_o, ph_o & 1);
    ++ph_o;
    tc_fence_after_sync();
    constexpr int ND = TW ? 16 : 32;  // output dims of a head written by this thread
#pragma unroll 1
    for (int h = 0; h < 4; ++h) {
      float o[ND];
      if (TW) tmem_ld16(tacc + 128 + 32 * h + 16 * tw, o);
      else tmem_ld32(tacc + 128 + 32 * h, o);
      tmem_wait_ld();
      if (ok) {
        const float inv = 1.f / (den_part[r * 4 + h] + (TW ? den_part[(128 + r) * 4 + h] : 0.f));
        uint8_t* dst = reinterpret_cast<uint8_t*>(O) + (size_t)tile * kTile +
                       (size_t)(4 * h + (TW ? 2 * tw : 0)) * 2048 + (size_t)r * 16;
#pragma unroll
        for (int i = 0; i < ND / 8; ++i)
          *reinterpret_cast<uint4*>(dst + i * 2048) = make_uint4(pack_bf16x2(o[8 * i] * inv, o[8 * i + 1] * inv),
                              pack_bf16x2(o[8 * i + 2] * inv, o[8 * i + 3] * inv),
                              pack_bf16x2(o[8 * i + 4] * inv, o[8 * i + 5] * inv),
                              pack_bf16x2(o[8 * i + 6] * inv, o[8 * i + 7] * inv));
      }
    }
    tc_fence_before_sync();
    __syncthreads();  // tiles + TMEM are reused by the next iteration
  }
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 256);
  }
}


// ---- S = 64 or 128: the bench shapes -------------------------------------------------------------------
// Same data flow as attention_tc_kernel<true>, specialised so that a thread's keys are exactly NB whole
// 32-column TMEM blocks (twin tw of row r owns keys [ray_lo + 32 NB tw, + 32 NB)):
//  * logits are read from TMEM once and stay in registers between the max and the exp pass;
//  * no per-key range tests; the 1/sqrt(32) scale, log2(e) and the max shift are one FFMA in front of ex2;
//  * the columns of P that belong to the tile's other ray (S = 64) are zero for every head and tile: they
//    are cleared once per CTA;
//  * K, Q_0 and V of the CTA's next tile are requested as soon as the last QK^T / PV of the current tile
//    has retired, so the loads overlap the last softmax and the write-out.
template <int NB>
__global__ void __launch_bounds__(256, 2)
attention_twin_kernel(const __nv_bfloat16* __restrict__ Q, const __nv_bfloat16* __restrict__ K,
                      const __nv_bfloat16* __restrict__ V, const float* __restrict__ nvalid, long long P,
                      __nv_bfloat16* __restrict__ O) {
  constexpr int S = 64 * NB;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* kt = smem;
  uint8_t* vt = smem + kTile;
  uint8_t* pt = smem + 2 * kTile;
  uint8_t* qt = smem + 3 * kTile;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 3 * kTile + kQSlice);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar_s = smem_u32(bars), bar_o = smem_u32(bars + 1);
  const uint32_t bar_k = smem_u32(bars + 2), bar_q = smem_u32(bars + 3), bar_v = smem_u32(bars + 5);
  if (tid == 0) {
    mbar_init(bar_s, 1); mbar_init(bar_o, 1); mbar_init(bar_k, 1); mbar_init(bar_q, 1); mbar_init(bar_v, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tacc = tmem_addr(tmem_base, (uint32_t)((warp & 3) * 32), 0);

  const int r = tid & 127, tw = tid >> 7, rw = warp & 3;
  const size_t roff = (size_t)(r >> 3) * 128 + (r & 7) * 16;
  const int ray_lo = (r / S) * S;
  const int k_lo = ray_lo + tw * 32 * NB;
  float* den_part = reinterpret_cast<float*>(bars + 8);  // [2][128][4]
  float* max_part = den_part + 2 * 128 * 4;              // [2][128]
  uint32_t ph_s = 0, ph_o = 0, ph_k = 0, ph_q = 0, ph_v = 0;
  const uint8_t* qimg = reinterpret_cast<const uint8_t*>(Q);
  const uint8_t* kimg = reinterpret_cast<const uint8_t*>(K);
  const uint8_t* vimg = reinterpret_cast<const uint8_t*>(V);

  if (NB == 1) {  // keys of the other ray of the tile: P = 0, never rewritten
#pragma unroll
    for (int kg = 0; kg < 16; ++kg)
      if ((kg * 8 < ray_lo || kg * 8 >= ray_lo + S) && (kg & 1) == tw)
        *reinterpret_cast<uint4*>(pt + roff + kg * 2048) = make_uint4(0u, 0u, 0u, 0u);
  }

  auto issue_qk = [&](int h) {
    mbar_wait(bar_q, ph_q & 1); ++ph_q;
    tc_fence_after_sync();
    if (elect_one()) {
      const uint32_t idesc = idesc_bf16_f32(128, 128);
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        mma_bf16_ss(tmem_base, smem_desc(smem_u32(qt) + (2 * ks) * 2048u, 2048u, 128u),
                    smem_desc(smem_u32(kt) + (4 * h + 2 * ks) * 2048u, 2048u, 128u), idesc, ks ? 1u : 0u);
      mma_commit(bar_s);
    }
    __syncwarp();
  };
  auto load_q = [&](long long tile, int h) {
    mbar_arrive_expect_tx(bar_q, (uint32_t)kQSlice);
    bulk_g2s(smem_u32(qt), qimg + (size_t)tile * kTile + (size_t)h * kQSlice, (uint32_t)kQSlice, bar_q);
  };
  auto load_k = [&](long long tile) {
    mbar_arrive_expect_tx(bar_k, (uint32_t)kTile);
    bulk_g2s(smem_u32(kt), kimg + (size_t)tile * kTile, (uint32_t)kTile, bar_k);
  };
  auto load_v = [&](long long tile) {
    mbar_arrive_expect_tx(bar_v, (uint32_t)kTile);
    bulk_g2s(smem_u32(vt), vimg + (size_t)tile * kTile, (uint32_t)kTile, bar_v);
  };

  const long long n_tiles = (P + 127) / 128;
  if (tid == 0 && (long long)blockIdx.x < n_tiles) {
    load_k(blockIdx.x);
    load_q(blockIdx.x, 0);
    load_v(blockIdx.x);
  }
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row = tile * 128 + r;
    const long long next = tile + gridDim.x;
    const bool ok = row < P;
    const bool q_valid = ok && nvalid[row] > 1.f;
    // exp(l / sqrt(32) - max) = 2^(l sc - max sc); a query row without two valid views attends uniformly
    const float sc = q_valid ? 0.17677669529663687f * 1.4426950408889634f : 0.f;
    if (warp == 0) {
      mbar_wait(bar_k, ph_k & 1); ++ph_k;
      issue_qk(0);
    }
#pragma unroll 1
    for (int h = 0; h < 4; ++h) {
      mbar_wait(bar_s, ph_s & 1);
      ++ph_s;
      tc_fence_after_sync();
      if (tid == 0) {
        if (h < 3) load_q(tile, h + 1);  // Q_h has been consumed
        else if (next < n_tiles) { load_k(next); load_q(next, 0); }  // and so has K
      }
      float l[NB][32];
#pragma unroll
      for (int b = 0; b < NB; ++b) tmem_ld32(tacc + k_lo + 32 * b, l[b]);
      tmem_wait_ld();
      float mx = l[0][0];
#pragma unroll
      for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int i = 0; i < 32; ++i) mx = fmaxf(mx, l[b][i]);
      max_part[tw * 128 + r] = mx;
      asm volatile("bar.sync %0, 64;" ::"r"(1 + rw) : "memory");
      mx = fmaxf(mx, max_part[(tw ^ 1) * 128 + r]);
      const float sh = mx * sc;
      // previous head's P V must be done before P is overwritten
      if (h > 0) { mbar_wait(bar_o, ph_o & 1); ++ph_o; }
      float den = 0.f;
#pragma unroll
      for (int b = 0; b < NB; ++b) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float e;
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaf(l[b][i], sc, -sh)));
          l[b][i] = e;
          den += e;
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 q;
          q.x = pack_bf16x2(l[b][8 * g], l[b][8 * g + 1]); q.y = pack_bf16x2(l[b][8 * g + 2], l[b][8 * g + 3]);
          q.z = pack_bf16x2(l[b][8 * g + 4], l[b][8 * g + 5]); q.w = pack_bf16x2(l[b][8 * g + 6], l[b][8 * g + 7]);
          *reinterpret_cast<uint4*>(pt + roff + ((k_lo >> 3) + 4 * b + g) * 2048) = q;
        }
      }
      den_part[(tw * 128 + r) * 4 + h] = den;  // 1 / sum applied when O is written out
      fence_proxy_async_smem();
      tc_fence_before_sync();
      __syncthreads();  // P complete; every thread is done reading logits_h
      if (warp == 0) {
        if (h == 0) { mbar_wait(bar_v, ph_v & 1); ++ph_v; }
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t idesc = idesc_bf16_f32_bmn(128, 32);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            mma_bf16_ss(tmem_base + 128 + 32 * h, smem_desc(smem_u32(pt) + ks * 4096u, 2048u, 128u),
                        smem_desc(smem_u32(vt) + (4 * h) * 2048u + ks * 256u, 128u, 2048u), idesc,
                        ks ? 1u : 0u);
          mma_commit(bar_o);
        }
        __syncwarp();
        if (h < 3) issue_qk(h + 1);
      }
    }
    mbar_wait(bar_o, ph_o & 1);
    ++ph_o;
    tc_fence_after_sync();
    if (tid == 0 && next < n_tiles) load_v(next);  // the last P V has retired: V is free
#pragma unroll 1
    for (int h = 0; h < 4; ++h) {
      float o[16];
      tmem_ld16(tacc + 128 + 32 * h + 16 * tw, o);
      tmem_wait_ld();
      if (ok) {
        const float inv = 1.f / (den_part[r * 4 + h] + den_part[(128 + r) * 4 + h]);
        uint8_t* dst = reinterpret_cast<uint8_t*>(O) + (size_t)tile * kTile + (size_t)(4 * h + 2 * tw) * 2048 +
                       (size_t)r * 16;
#pragma unroll
        for (int i = 0; i < 2; ++i)
          *reinterpret_cast<uint4*>(dst + i * 2048) = make_uint4(pack_bf16x2(o[8 * i] * inv, o[8 * i + 1] * inv),
                              pack_bf16x2(o[8 * i + 2] * inv, o[8 * i + 3] * inv),
                              pack_bf16x2(o[8 * i + 4] * inv, o[8 * i + 5] * inv),
                              pack_bf16x2(o[8 * i + 6] * inv, o[8 * i + 7] * inv));
      }
    }
    tc_fence_before_sync();
    __syncthreads();  // P, den_part and TMEM are reused by the next iteration
  }
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 256);
  }
}

}  // namespace

bool attention_tc_supported(int S) { return S >= 1 && S <= 128 && (128 % S) == 0; }

int launch_attention_tc(const __nv_bfloat16* Q, const __nv_bfloat16* K, const __nv_bfloat16* V,
                        const float* nvalid, long long P, int S, __nv_bfloat16* O, cudaStream_t st) {
  if (P == 0) return DYN_OK;
  int dev = 0, sms = 148;
  DYN_CUDA(cudaGetDevice(&dev));
  DYN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long n_tiles = (P + 127) / 128;
  const int grid = (int)(n_tiles < 2 * sms ? n_tiles : 2 * sms);
  const int smem = kSmemAttn;
  ProfScope prof(PROF_ATTENTION, st);
  static const bool generic = getenv("DYN_ATTENTION") && !strcmp(getenv("DYN_ATTENTION"), "generic");
  static bool attr_done = false;  // one device per process (torch.distributed: one rank per GPU)
  if (!attr_done) {
    DYN_CUDA(cudaFuncSetAttribute(attention_twin_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    DYN_CUDA(cudaFuncSetAttribute(attention_twin_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    DYN_CUDA(cudaFuncSetAttribute(attention_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    DYN_CUDA(cudaFuncSetAttribute(attention_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done = true;
  }
  if (S == 64 && !generic) {
    attention_twin_kernel<1><<<grid, 256, smem, st>>>(Q, K, V, nvalid, P, O);
  } else if (S == 128 && !generic) {
    attention_twin_kernel<2><<<grid, 256, smem, st>>>(Q, K, V, nvalid, P, O);
  } else if (S % 64 == 0) {  // twin warps
    attention_tc_kernel<true><<<grid, 256, smem, st>>>(Q, K, V, nvalid, P, S, O);
  } else {
    attention_tc_kernel<false><<<grid, 128, smem, st>>>(Q, K, V, nvalid, P, S, O);
  }
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // namespace dyn
