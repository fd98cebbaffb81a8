// Shared machinery of the fused tcgen05 kernels (view_twin3.cu, chains_twin.cu, chains_fused.cu):
// smem budget constants, fast activations, A-tile stores, view-group shuffles,
// the table-driven weight producer and MMA issuer, and the host-side packing of
// weight chunks into UMMA images.
#pragma once
#include <vector>

#include "nets_fused.cuh"
#include "tc.cuh"

namespace dyn {
namespace fe {

using namespace tc;

constexpr int kRing = 4;
constexpr int kStageBytes = 16384;
constexpr int kATileBytes = 69632;  // 128 rows x 272 cols bf16 (34 k-groups: geometry_fc.0 has K = 257)
// barrier slots inside the fused kernels: [0..3] w_full, [4..7] w_empty, [8] a_ready, [9] acc_full

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float elu_fast(float x) {
  float e = ex2f(x * 1.4426950408889634f);
  return x > 0.f ? x : e - 1.f;
}
// ELU on the exp2 scale: x2 = log2(e) * x in, log2(e) * ELU(x) out (4 instructions; the producing layer's
// weights and folded bias carry the log2 e, the consuming layer's weights the ln 2)
__device__ __forceinline__ float elu_log2(float x2) {
  const float e = ex2f(x2);
  return x2 > 0.f ? x2 : fmaf(e, 1.4426950408889634f, -1.4426950408889634f);
}
// ELU in true units from an accumulator on the exp2 scale (x2 = log2(e) * x): 4 instructions
__device__ __forceinline__ float elu_from_log2(float x2) {
  const float e = ex2f(x2);
  return x2 > 0.f ? x2 * 0.6931471805599453f : e - 1.f;
}
__device__ __forceinline__ float sigmoid_fast(float x) {
  return __frcp_rn(1.f + ex2f(-x * 1.4426950408889634f));
}

// tcgen05.wait::ld that carries a data dependency on the 16 destination registers of the load it waits for (so no
// use of them can be scheduled above it)
__device__ __forceinline__ void tmem_wait_ld_dep16(float* v) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                 "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
               :
               : "memory");
}

// Software-pipelined accumulator read-out: NH half-blocks of 16 TMEM columns; the load of half h + 1 is in flight
// while fn(h, values) processes half h (TMEM reads run at 64 B/clk: a 32-column load of one warp occupies the port
// for 64 cycles, and eight row warps per CTA queue on it).  colf(h) = TMEM column of half h.
template <int NH, class ColFn, class Fn>
__device__ __forceinline__ void tmem_pipe16(uint32_t tacc, ColFn colf, Fn fn) {
  float buf[2][16];
  tmem_ld16(tacc + colf(0), buf[0]);
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    tmem_wait_ld_dep16(buf[h & 1]);
    if (h + 1 < NH) tmem_ld16(tacc + colf(h + 1), buf[(h + 1) & 1]);
    fn(h, buf[h & 1]);
  }
}

// 8 consecutive columns [c0, c0+8) of this thread's row -> one 16-byte store
__device__ __forceinline__ void store8(uint8_t* arow, int c0, const float* v) {
  uint4 q;
  q.x = pack_bf16x2(v[0], v[1]);
  q.y = pack_bf16x2(v[2], v[3]);
  q.z = pack_bf16x2(v[4], v[5]);
  q.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(arow + (c0 >> 3) * 2048) = q;
}

// PE with frequencies 2^k via angle doubling: out = [x(D), cos(2^k x)(NF*D), sin(2^k x)(NF*D)]
template <int D, int NF>
__device__ __forceinline__ void pe_pow2(const float* x, float* out) {
#pragma unroll
  for (int d = 0; d < D; ++d) {
    out[d] = x[d];
    float s, c;
    __sincosf(x[d], &s, &c);
#pragma unroll
    for (int k = 0; k < NF; ++k) {
      out[D + k * D + d] = c;
      out[D + NF * D + k * D + d] = s;
      float s2 = 2.f * s * c, c2 = 1.f - 2.f * s * s;
      s = s2; c = c2;
    }
  }
}

template <int VP>
__device__ __forceinline__ float group_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  if (VP == 16) v += __shfl_xor_sync(0xffffffffu, v, 8);
  return v;
}
template <int VP>
__device__ __forceinline__ float group_min(float v) {
  v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 4));
  if (VP == 16) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, 8));
  return v;
}

// one reduce-scatter step over N values: lanes with `bit` set keep the upper half
template <int N>
__device__ __forceinline__ void rs_step(const float* in, float* out, bool upper, int xr) {
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    float send = upper ? in[i] : in[N / 2 + i];
    float keep = upper ? in[N / 2 + i] : in[i];
    out[i] = keep + __shfl_xor_sync(0xffffffffu, send, xr);
  }
}


// "Tile image": how bf16 activations travel between fused kernels through HBM.  Rows are grouped in
// tiles of 128 and stored exactly as the consumer's UMMA A operand sits in shared memory (K-major
// 8x8 core matrices): element (row r, column k) of a tile with KG 8-column groups lives at byte
//   tile * KG * 2048 + (k / 8) * 2048 + (r % 128) * 16 + (k % 8) * 2.
// The producer's per-row 16-byte stores are therefore warp-coalesced (32 rows x 16 B = 512 B), and
// the consumer lands a whole operand block with ONE cp.async.bulk instead of per-thread loads.
__host__ __device__ __forceinline__ size_t tile_image_off(long long row, int kgroup, int kgroups) {
  return (size_t)(row >> 7) * (size_t)kgroups * 2048u + (size_t)kgroup * 2048u + (size_t)(row & 127) * 16u;
}
__host__ __device__ __forceinline__ size_t tile_image_bytes(long long rows, int kgroups) {
  return (size_t)((rows + 127) >> 7) * (size_t)kgroups * 2048u;
}

// fp32 companion of the tile image for per-point vectors that stay fp32 (residual stream g2, the
// blending head's per-point term GW): 128 columns in groups of 4 floats, element (row r, column c)
// of a 128-row tile at byte  tile * 65536 + (c / 4) * 2048 + (r % 128) * 16 + (c % 4) * 4,
// so that both the producer's and the consumer's per-row float4 accesses are warp-coalesced.
__host__ __device__ __forceinline__ size_t tile_f32_off(long long row, int col4group) {
  return (size_t)(row >> 7) * 65536u + (size_t)col4group * 2048u + (size_t)(row & 127) * 16u;
}

// The chunk table is staged into shared memory once per CTA: the producer and the issuer
// read one entry per chunk on their critical path (a global load there costs an L2 round trip
// per chunk and was the bottleneck of the MMA issue thread).
constexpr int kMaxChunks = 160;
__device__ __forceinline__ void stage_chunks(FusedChunk* s, const FusedChunk* __restrict__ g, int n) {
  static_assert(sizeof(FusedChunk) == 16, "FusedChunk is copied as uint4");
  const uint4* src = reinterpret_cast<const uint4*>(g);
  uint4* dst = reinterpret_cast<uint4*>(s);
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// ---- control warps (one elected lane each) -------------------------------------
// barrier slots: [0..3] w_full, [4..7] w_empty, [8] a_ready(tile0), [9] acc_full(tile0),
//                [10] a_ready(tile1), [11] acc_full(tile1)
// Two schedules:
//   lock-step (PP = false): both 128-row tiles consume every weight chunk together
//     (weights stream once per 256 rows); one a_ready (256 arrivals) / acc_full pair.
//   ping-pong (PP = true): per ROUND (chunks from a wait-flag to a last-flag) tile 0
//     then tile 1, each with its own barriers (128 arrivals), so the MMA of one tile
//     overlaps the epilogue of the other; weights stream twice.
// generic layout for a ring of `ring` slots: [0,ring) w_full, [ring,2 ring) w_empty, then per tile a_ready, acc_full
__device__ __forceinline__ uint32_t bar_aready(uint32_t bar0, int tile, int ring = kRing) { return bar0 + 8u * (2 * ring + 2 * tile); }
__device__ __forceinline__ uint32_t bar_acc(uint32_t bar0, int tile, int ring = kRing) { return bar0 + 8u * (2 * ring + 1 + 2 * tile); }

// `arrivals` = row threads per 128-row tile (128, or 256 in the twin-warp kernels)
__device__ __forceinline__ void init_barriers(uint32_t bar0, bool pp, int arrivals = 128, int ring = kRing) {
  for (int i = 0; i < ring; ++i) { mbar_init(bar0 + 8u * i, 1); mbar_init(bar0 + 8u * (ring + i), 1); }
  mbar_init(bar_aready(bar0, 0, ring), pp ? arrivals : 2 * arrivals);
  mbar_init(bar_acc(bar0, 0, ring), 1);
  mbar_init(bar_aready(bar0, 1, ring), arrivals);
  mbar_init(bar_acc(bar0, 1, ring), 1);
  mbar_fence_init();
}

__device__ __forceinline__ int round_end(const FusedChunk* __restrict__ chunks, int c0, int nchunks) {
  int c = c0;
  while (c < nchunks && !(chunks[c].flags & 2)) ++c;
  return c + 1 < nchunks ? c + 1 : nchunks;
}

// One thread sustains ~40 B/clk of cp.async.bulk traffic however many copies it keeps in flight, two
// threads ~79 B/clk, three ~100 B/clk (profiles/scripts/tma_rate.cu, profiles/r02_view_kernels.md), while
// a layer at the full MMA rate consumes 64 B/clk of weights: `nlanes` lanes of the producer warp share
// the chunk stream round-robin (lane p issues the chunks with cnt % nlanes == p; RING % nlanes == 0, so
// a lane always refills the same ring slots).
template <bool PP, int RING = kRing, int STAGE = kStageBytes>
__device__ __forceinline__ void producer_loop(const FusedChunk* __restrict__ chunks, int nchunks,
                                              const void* wimg, int n_iter, uint8_t* ring, uint32_t bar0,
                                              uint32_t lane = 0, uint32_t nlanes = 1) {
  const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(wimg);
  uint32_t cnt = 0;
  for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
    for (int c0 = 0; c0 < nchunks;) {
      const int c1 = PP ? round_end(chunks, c0, nchunks) : nchunks;
      for (int rep = 0; rep < (PP ? 2 : 1); ++rep) {
        for (int c = c0; c < c1; ++c, ++cnt) {
          if (cnt % nlanes != lane) continue;
          const uint32_t st = cnt % RING;
          if (cnt >= RING) mbar_wait(bar0 + 8u * (RING + st), ((cnt / RING) - 1) & 1);
          const FusedChunk ch = chunks[c];
          mbar_arrive_expect_tx(bar0 + 8u * st, ch.bytes);
          bulk_g2s(smem_u32(ring + st * STAGE), wsrc + ch.off, ch.bytes, bar0 + 8u * st);
        }
      }
      c0 = c1;
    }
  }
}

// Called by ALL 32 lanes of the issuer warp (converged).
// FusedChunk.flags: 1 = wait for a_ready before this chunk, 2 = last chunk of a
// round (commit acc_full), 4 = wait for the second operand barrier (one-tile kernels: the
// a_ready slot of tile 1) before this chunk, 8 = first k-step overwrites D (start of a layer);
// d_col = accumulator column offset inside the tile's 256-column TMEM region.
// NT = 128-row tiles per CTA (1 or 2), RING = weight-ring slots in use.
template <bool PP, int NT = 2, int RING = kRing, int STAGE = kStageBytes>
__device__ __forceinline__ void issuer_loop(const FusedChunk* __restrict__ chunks, int nchunks, int n_iter,
                                            uint8_t* smem, uint8_t* ring, uint32_t bar0,
                                            uint32_t tmem_base, int a_tile_bytes = kATileBytes,
                                            long long* dbg = nullptr) {
  // Entered by the whole (converged) warp; ONE elected lane then runs the loop alone, so every
  // address / descriptor stays in uniform registers and no per-chunk warp re-convergence is needed.
  if (elect_one()) {
    uint32_t cnt = 0, a_cnt[2] = {0, 0}, a2_cnt = 0;
    long long t_a = 0, t_w = 0, t_begin = clock64();
    const uint32_t a_addr[2] = {smem_u32(smem), smem_u32(smem + a_tile_bytes)};
    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      for (int c0 = 0; c0 < nchunks;) {
        const int c1 = PP ? round_end(chunks, c0, nchunks) : nchunks;
        for (int rep = 0; rep < (PP ? 2 : 1); ++rep) {
          for (int c = c0; c < c1; ++c, ++cnt) {
            const FusedChunk ch = chunks[c];
            long long t0 = dbg ? clock64() : 0;
            if (ch.flags & 1) {
              mbar_wait(bar_aready(bar0, PP ? rep : 0, RING), a_cnt[PP ? rep : 0] & 1);
              ++a_cnt[PP ? rep : 0];
            }
            if (!PP && NT == 1 && (ch.flags & 4)) {  // second operand barrier of a two-sub-round layer
              mbar_wait(bar_aready(bar0, 1, RING), a2_cnt & 1);
              ++a2_cnt;
            }
            long long t1 = dbg ? clock64() : 0;
            const uint32_t st = cnt % RING;
            mbar_wait(bar0 + 8u * st, (cnt / RING) & 1);
            tc_fence_after_sync();
            long long t2 = 0;
            if (dbg) {
              t2 = clock64();
              t_a += t1 - t0;
              t_w += t2 - t1;
            }
            const uint32_t idesc = idesc_bf16_f32(128, ch.npad);
            const uint32_t w_addr = smem_u32(ring + st * STAGE);
            const uint32_t lbo_b = (uint32_t)ch.npad * 16u;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
              if (PP && t != rep) continue;
              const uint32_t aa = a_addr[t] + (uint32_t)ch.a_kgroup * 2048u;
              for (int ks = 0; ks < ch.ksteps; ++ks) {
                mma_bf16_ss(tmem_base + t * 256 + ch.d_col, smem_desc(aa + ks * 4096u, 2048u, 128u),
                            smem_desc(w_addr + ks * 2u * lbo_b, lbo_b, 128u), idesc,
                            ((ch.flags & 8) && ks == 0) ? 0u : 1u);
              }
            }
            mma_commit(bar0 + 8u * (RING + st));
            if (ch.flags & 2) mma_commit(bar_acc(bar0, PP ? rep : 0, RING));
            if (dbg && blockIdx.x == 0 && cnt < 120) {
              dbg[8 + 4 * cnt + 0] = t0; dbg[8 + 4 * cnt + 1] = t1;
              dbg[8 + 4 * cnt + 2] = t2; dbg[8 + 4 * cnt + 3] = clock64();
            }
          }
        }
        c0 = c1;
      }
    }
    if (dbg != nullptr && blockIdx.x == 0) {
      dbg[0] = clock64() - t_begin;  // issuer lifetime
      dbg[1] = t_a;                  // waiting for A operands (epilogues)
      dbg[2] = t_w;                  // waiting for weight chunks (ring)
    }
  }
  __syncwarp();
}

// ---- host side: weight images + chunk table ------------------------------------
inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN
  uint32_t lsb = (u >> 16) & 1u;
  u += 0x7fffu + lsb;  // round to nearest even
  return (uint16_t)(u >> 16);
}

struct HostLayer {
  const float* W;  // host fp32 [*, Kw]
  int N, Kw, Npad, Kpad;
  std::vector<int> colmap;  // size Kpad: weight column, -1 (zero), or kBiasHi / kBiasLo
  // bias folded into the MMA: the operand carries 1.0 in the kBiasHi and kBiasLo columns and the image
  // holds bf16(b) and bf16(b - bf16(b)) there (error 2^-17 |b|); `scale` multiplies weights and bias
  // (log2 e for layers whose ELU is evaluated on the exp2 scale, ln 2 for their consumers)
  const float* bias = nullptr;
  float scale = 1.f;
  float bias_scale = -1.f;  // < 0: same as `scale` (differs when the layer CONSUMES a log2-scaled operand
                            // and PRODUCES an exp2-scale accumulator: weights x ln2 x log2e = 1, bias x log2e)
  std::vector<float> colscale;  // optional, size Kpad: extra factor per OPERAND column (operand tiles that mix
                                // exp2-scale activations with true-scale encodings)
};
constexpr int kBiasHi = -2, kBiasLo = -3;
inline float bf2f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

inline void append_layer(const HostLayer& L, std::vector<uint8_t>& img, std::vector<FusedChunk>& tab,
                         int d_col = 0, int a_kgroup0 = 0, int first_flags = 9, bool last = true,
                         int stage_bytes = kStageBytes) {
  int steps_per_chunk = stage_bytes / (L.Npad * 32);
  if (steps_per_chunk > 8) steps_per_chunk = 8;
  const int ksteps_total = L.Kpad / 16;
  for (int k0 = 0; k0 < ksteps_total; k0 += steps_per_chunk) {
    const int ks = (ksteps_total - k0) < steps_per_chunk ? (ksteps_total - k0) : steps_per_chunk;
    FusedChunk ch;
    ch.off = (uint32_t)img.size();
    ch.bytes = (uint32_t)(L.Npad * 32 * ks);
    ch.npad = (uint16_t)L.Npad;
    ch.ksteps = (uint8_t)ks;
    ch.flags = (uint8_t)((k0 == 0 ? first_flags : 0) | ((last && k0 + ks >= ksteps_total) ? 2 : 0));
    ch.a_kgroup = (uint16_t)(a_kgroup0 + k0 * 2);
    ch.d_col = (uint16_t)d_col;
    img.resize(img.size() + ch.bytes, 0);
    uint16_t* dst = reinterpret_cast<uint16_t*>(img.data() + ch.off);
    for (int n = 0; n < L.Npad; ++n)
      for (int kk = 0; kk < ks * 16; ++kk) {
        const int col = L.colmap[k0 * 16 + kk];
        float val = 0.f;
        if (n < L.N) {
          if (col >= 0) {
            val = L.W[(size_t)n * L.Kw + col] * L.scale * (L.colscale.empty() ? 1.f : L.colscale[k0 * 16 + kk]);
          } else if (L.bias != nullptr && (col == kBiasHi || col == kBiasLo)) {
            const float b = L.bias[n] * (L.bias_scale >= 0.f ? L.bias_scale : L.scale), hi = bf2f(f2bf(b));
            val = col == kBiasHi ? hi : b - hi;
          }
        }
        dst[tile_off((uint32_t)L.Npad, (uint32_t)n, (uint32_t)kk) / 2] = f2bf(val);
      }
    tab.push_back(ch);
  }
}

// A layer issued in SUB-ROUNDS: `plan[r]` lists the runs (first k-step, number of k-steps) of operand columns
// that sub-round r consumes; the issuer waits for one operand arrival round per sub-round (chunk flag 1) and
// signals the epilogue only after the last one (flag 2).  The row warps arrive after every block of operand
// columns they finish, so the k-steps over finished columns overlap the epilogue of the remaining ones.
// Chunk c of a run starting at k-step k0 reads the operand tile at k-group a_kgroup0 + 2 * (k0 + ...).
using LayerPlan = std::vector<std::vector<std::pair<int, int>>>;
inline void append_layer_plan(const HostLayer& L, std::vector<uint8_t>& img, std::vector<FusedChunk>& tab,
                              int d_col, int a_kgroup0, const LayerPlan& plan, int stage_bytes = kStageBytes) {
  int steps_per_chunk = stage_bytes / (L.Npad * 32);
  if (steps_per_chunk > 8) steps_per_chunk = 8;
  bool first_chunk = true;
  for (size_t r = 0; r < plan.size() && r < 2; ++r) {  // at most two sub-rounds (two operand barriers)
    bool first_of_round = true;
    for (size_t q = 0; q < plan[r].size(); ++q) {
      const int run0 = plan[r][q].first, run1 = run0 + plan[r][q].second;
      for (int k0 = run0; k0 < run1; k0 += steps_per_chunk) {
        const int ks = (run1 - k0) < steps_per_chunk ? (run1 - k0) : steps_per_chunk;
        const bool last = r + 1 == plan.size() && q + 1 == plan[r].size() && k0 + ks >= run1;
        FusedChunk ch;
        ch.off = (uint32_t)img.size();
        ch.bytes = (uint32_t)(L.Npad * 32 * ks);
        ch.npad = (uint16_t)L.Npad;
        ch.ksteps = (uint8_t)ks;
        // sub-round 0 waits on the operand barrier (flag 1), sub-round 1 on the SECOND operand barrier (flag 4):
        // a row thread arrives on each of them exactly once per layer -- with a single barrier a fast thread's
        // second arrival could complete the phase that a slow thread has not reached yet
        ch.flags = (uint8_t)((first_of_round ? (r == 0 ? 1 : 4) : 0) | (first_chunk ? 8 : 0) | (last ? 2 : 0));
        ch.a_kgroup = (uint16_t)(a_kgroup0 + k0 * 2);
        ch.d_col = (uint16_t)d_col;
        img.resize(img.size() + ch.bytes, 0);
        uint16_t* dst = reinterpret_cast<uint16_t*>(img.data() + ch.off);
        const float bs = L.bias_scale >= 0.f ? L.bias_scale : L.scale;
        for (int n = 0; n < L.Npad; ++n)
          for (int kk = 0; kk < ks * 16; ++kk) {
            const int col = L.colmap[k0 * 16 + kk];
            float val = 0.f;
            if (n < L.N) {
              if (col >= 0) {
                val = L.W[(size_t)n * L.Kw + col] * L.scale * (L.colscale.empty() ? 1.f : L.colscale[k0 * 16 + kk]);
              } else if (L.bias != nullptr && (col == kBiasHi || col == kBiasLo)) {
                const float b = L.bias[n] * bs, hi = bf2f(f2bf(b));
                val = col == kBiasHi ? hi : b - hi;
              }
            }
            dst[tile_off((uint32_t)L.Npad, (uint32_t)n, (uint32_t)kk) / 2] = f2bf(val);
          }
        tab.push_back(ch);
        first_of_round = false;
        first_chunk = false;
      }
    }
  }
}

inline std::vector<int> identity_map(int K, int Kpad) {
  std::vector<int> m(Kpad, -1);
  for (int i = 0; i < K; ++i) m[i] = i;
  return m;
}


}  // namespace fe
}  // namespace dyn
