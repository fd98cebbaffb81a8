// The MotionMLP as one fused tcgen05 chain (row-local: no cross-row reduction inside it), built on
// fused_engine.cuh:
//
//   motion_fused_kernel : PE(xyzt) -> 8 x (256, ReLU) with skip -> 18 coeffs
//                         (mlp_network.py:605-618 + render_ray.py:459-472)
//
// 256 rows per iteration (two M=128 UMMA tiles), one row per thread in warps 0-7, the MMA issuer in
// warp 8 and the weight producer in warp 9.  The aggregation nets' row-local chains are in chains_twin.cu.
// Also here: the host-only unit-test hooks behind dyn_debug_pack_layer / dyn_debug_tile_image_off.
#include "fused_engine.cuh"
#include "nets.cuh"

namespace dyn {

using namespace tc;
using namespace fe;

namespace {

// common prologue: barriers + TMEM; returns the TMEM base address
__device__ __forceinline__ uint32_t fused_prologue(uint64_t* bars, uint32_t* tmem_slot, bool pp) {
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  if (tid == 0) init_barriers(bar0, pp);
  if (warp == 8) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  return *tmem_slot;
}
__device__ __forceinline__ void fused_teardown(uint32_t tmem_base) {
  __syncthreads();
  if ((threadIdx.x >> 5) == 8) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}
// `bt` = barrier tile: the thread's tile in ping-pong kernels, 0 in lock-step kernels
__device__ __forceinline__ void operand_ready(uint32_t bar0, int bt) {
  fence_proxy_async_smem();
  tc_fence_before_sync();
  mbar_arrive(bar_aready(bar0, bt));
}
__device__ __forceinline__ void wait_acc(uint32_t bar0, int bt, uint32_t& acc_cnt) {
  mbar_wait(bar_acc(bar0, bt), acc_cnt & 1);
  ++acc_cnt;
  tc_fence_after_sync();
}

// ReLU(acc + bias) of `ncols` accumulator columns -> bf16 operand columns [0, ncols)
__device__ __forceinline__ void relu_cols_to_A(uint8_t* arow, uint32_t tacc, int ncols, const float* bias) {
#pragma unroll 1
  for (int cb = 0; cb < ncols; cb += 32) {
    float acc[32];
    tmem_ld32(tacc + cb, acc);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = fmaxf(acc[i] + bias[cb + i], 0.f);
#pragma unroll
    for (int g = 0; g < 4; ++g) store8(arow, cb + 8 * g, acc + 8 * g);
  }
}

// ---------------------------------------------------------------------------
// MotionMLP
// ---------------------------------------------------------------------------
// operand column order of PE(xyzt): for k in 0..15: [cos(f_k x)(4) | sin(f_k x)(4)], then [x(4) | 0 x 12]
__device__ __forceinline__ void motion_operand(uint8_t* arow, const float* x4, bool valid) {
  // f_k = 1 + k * 16/15 (torch.linspace(1, 17, 16)); angle-addition recurrence
  const float delta = 16.f / 15.f;
  float c[4], s[4], cd[4], sd[4];
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    __sincosf(x4[d], &s[d], &c[d]);
    __sincosf(x4[d] * delta, &sd[d], &cd[d]);
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    float o[8];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      o[d] = valid ? c[d] : 0.f;
      o[4 + d] = valid ? s[d] : 0.f;
      const float cn = c[d] * cd[d] - s[d] * sd[d];
      const float sn = s[d] * cd[d] + c[d] * sd[d];
      c[d] = cn; s[d] = sn;
    }
    store8(arow, 8 * k, o);
  }
  float o[8] = {valid ? x4[0] : 0.f, valid ? x4[1] : 0.f, valid ? x4[2] : 0.f, valid ? x4[3] : 0.f,
                0.f, 0.f, 0.f, 0.f};
  store8(arow, 128, o);
  float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  store8(arow, 136, z);
}

__global__ void __launch_bounds__(320, 1) motion_fused_kernel(const __grid_constant__ MotionFusedArgs a) {
  constexpr bool kPP = false;  // MMA-bound ReLU chain: share every weight chunk between the tiles
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem + 2 * kATileBytes;
  float* cst = reinterpret_cast<float*>(ring + kRing * kStageBytes);  // 8 x 256 biases + 32
  uint64_t* bars = reinterpret_cast<uint64_t*>(cst + 2304);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  __shared__ __align__(16) FusedChunk s_tab[kMaxChunks];
  stage_chunks(s_tab, a.chunks, a.nchunks);
  for (int i = tid; i < 2048; i += blockDim.x) cst[i] = a.params[a.o_bias[i >> 8] + (i & 255)];
  if (tid < 32) cst[2048 + tid] = tid < a.ncoef ? a.params[a.o_bias[8] + tid] : 0.f;
  const uint32_t tmem_base = fused_prologue(bars, tmem_slot, kPP);
  const int n_iter = (int)((a.N + 255) / 256);

  if (warp == 9) {
    if ((tid & 31) < a.producers) producer_loop<kPP>(s_tab, a.nchunks, a.wimg, n_iter, ring, bar0, tid & 31, a.producers);
  } else if (warp == 8) {
    issuer_loop<kPP>(s_tab, a.nchunks, n_iter, smem, ring, bar0, tmem_base);
  } else {
    const int tile = tid >> 7, r = tid & 127;
    const int bt = kPP ? tile : 0;
    uint8_t* arow = smem + tile * kATileBytes + (r >> 3) * 128 + (r & 7) * 16;
    const uint32_t tacc = tmem_addr(tmem_base, (uint32_t)((warp & 3) * 32), (uint32_t)(tile * 256));
    uint32_t acc_cnt = 0;
    for (int it = blockIdx.x; it < n_iter; it += gridDim.x) {
      const long long row = (long long)it * 256 + tid;
      const bool valid = row < a.N;
      float x4[4] = {0.f, 0.f, 0.f, a.time};
      if (valid) {
        const float* src = a.x + row * a.ldx;
        x4[0] = src[0]; x4[1] = src[1]; x4[2] = src[2];
        if (a.time_is_column) x4[3] = src[3];
      }
      motion_operand(arow, x4, valid);
      operand_ready(bar0, bt);
      for (int l = 0; l < 5; ++l) {  // pts_linears.0 .. 4
        wait_acc(bar0, bt, acc_cnt);
        relu_cols_to_A(arow, tacc, 256, cst + 256 * l);
        operand_ready(bar0, bt);
      }
      // pts_linears.5 on cat([input_pts, h]): h part consumed first, then the
      // operand tile is re-filled with PE(xyzt) and the MMA keeps accumulating
      wait_acc(bar0, bt, acc_cnt);
      motion_operand(arow, x4, valid);
      operand_ready(bar0, bt);
      for (int l = 5; l < 8; ++l) {  // epilogues of pts_linears.5 .. 7
        wait_acc(bar0, bt, acc_cnt);
        relu_cols_to_A(arow, tacc, 256, cst + 256 * l);
        operand_ready(bar0, bt);
      }
      // coeff_linear (18 of 32 columns), zero the last samples of each ray
      wait_acc(bar0, bt, acc_cnt);
      float acc[32];
      tmem_ld32(tacc, acc);
      tmem_wait_ld();
      if (valid) {
        const bool zero = a.S > 0 && (int)(row % a.S) >= a.S - a.n_last;
        float* dst = a.coeff + row * a.ncoef;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < a.ncoef) dst[i] = zero ? 0.f : (acc[i] + cst[2048 + i]);
      }
      tc_fence_before_sync();
    }
  }
  fused_teardown(tmem_base);
}

constexpr int kSmemChain = 2 * kATileBytes + kRing * kStageBytes + 2304 * 4 + 256;

template <class K, class A>
int launch_chain(K kernel, const A& args, long long rows, cudaStream_t st) {
  int dev = 0, sms = 148;
  DYN_CUDA(cudaGetDevice(&dev));
  DYN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long n_iter = (rows + 255) / 256;
  const int grid = (int)(n_iter < sms ? n_iter : sms);
  if (grid == 0) return DYN_OK;
  DYN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemChain));
  kernel<<<grid, 320, kSmemChain, st>>>(args);
  DYN_LAUNCH_CHECK();
  return DYN_OK;
}

}  // namespace

// ---------------------------------------------------------------------------
// host: chunk tables
// ---------------------------------------------------------------------------
static void upload(std::vector<uint8_t>& img, std::vector<FusedChunk>& tab, char*& cursor, size_t& left,
                   ChainImage* out, cudaStream_t st, int* rc) {
  const size_t img_bytes = (img.size() + 255) & ~(size_t)255;
  const size_t need = img_bytes + ((tab.size() * sizeof(FusedChunk) + 255) & ~(size_t)255);
  if (need > left) { *rc = fail(DYN_E_INVALID, "fused chain images need %zu bytes, have %zu", need, left); return; }
  cudaMemcpyAsync(cursor, img.data(), img.size(), cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(cursor + img_bytes, tab.data(), tab.size() * sizeof(FusedChunk), cudaMemcpyHostToDevice, st);
  cudaStreamSynchronize(st);
  out->img = cursor;
  out->tab = reinterpret_cast<const FusedChunk*>(cursor + img_bytes);
  out->nchunks = (int)tab.size();
  if (tab.size() > (size_t)kMaxChunks) { *rc = fail(DYN_E_INVALID, "chunk table too long (%zu)", tab.size()); return; }
  cursor += need;
  left -= need;
  img.clear();
  tab.clear();
}

// host-only unit-test hooks behind dyn_debug_pack_layer / dyn_debug_tile_image_off
int debug_pack_layer(const float* W, const float* bias, int N, int Kw, int Npad, int Kpad, const int* colmap,
                     float scale, int stage_bytes, void* out_img, size_t out_bytes, size_t* img_bytes,
                     int* nchunks) {
  if (N < 1 || Npad < N || (Npad % 16) != 0 || Npad > 256 || (Kpad % 16) != 0 || Kpad < 16 || Kw < 1 ||
      stage_bytes < Npad * 32)
    return fail(DYN_E_INVALID, "dyn_debug_pack_layer: bad shape N=%d Npad=%d Kpad=%d stage=%d", N, Npad, Kpad,
                stage_bytes);
  HostLayer L;
  L.W = W; L.N = N; L.Kw = Kw; L.Npad = Npad; L.Kpad = Kpad;
  L.colmap.assign(colmap, colmap + Kpad);
  for (int c : L.colmap)
    if (c >= Kw || c < kBiasLo) return fail(DYN_E_INVALID, "dyn_debug_pack_layer: colmap entry %d out of range", c);
  L.bias = bias; L.scale = scale;
  std::vector<uint8_t> img;
  std::vector<FusedChunk> tab;
  append_layer(L, img, tab, 0, 0, 9, true, stage_bytes);
  *img_bytes = img.size();
  *nchunks = (int)tab.size();
  if (img.size() > out_bytes) return fail(DYN_E_INVALID, "dyn_debug_pack_layer: image needs %zu bytes", img.size());
  memcpy(out_img, img.data(), img.size());
  return DYN_OK;
}
size_t debug_tile_image_off(long long row, int kgroup, int kgroups) { return tile_image_off(row, kgroup, kgroups); }

size_t fused_chain_bytes(int kind) { return kind == DYN_NET_MOTION ? (size_t)(1280 * 1024) : 0; }

int fused_chain_build(dyn_net* n, const float* P, void* dst_dev, size_t dst_bytes, cudaStream_t st) {
  if (n->kind != DYN_NET_MOTION) return DYN_OK;
  std::vector<uint8_t> img;
  std::vector<FusedChunk> tab;
  char* cur = reinterpret_cast<char*>(dst_dev);
  size_t left = dst_bytes;
  int rc = DYN_OK;
  auto add = [&](const LinearP& l, int N, int Npad, int Kpad, std::vector<int> map, int first_flags = 9) {
    HostLayer L;
    L.W = P + l.w; L.N = N; L.Kw = l.in; L.Npad = Npad; L.Kpad = Kpad;
    L.colmap = std::move(map);
    append_layer(L, img, tab, 0, 0, first_flags, true);
  };
  const MotionLayout& L = n->ml;
  // operand order: k-major [cos f_k (4) | sin f_k (4)] x 16, then x(4): weight column of each
  std::vector<int> pe(144, -1);
  for (int k = 0; k < 16; ++k)
    for (int d = 0; d < 4; ++d) { pe[8 * k + d] = 4 + 4 * k + d; pe[8 * k + 4 + d] = 68 + 4 * k + d; }
  for (int d = 0; d < 4; ++d) pe[128 + d] = d;
  add(L.pts[0], 256, 256, 144, pe);
  for (int i = 1; i < 5; ++i) add(L.pts[i], 256, 256, 256, identity_map(256, 256));
  {  // pts_linears.5: input cat([pe(132), h(256)]) -> h part first, then the pe part accumulates
    std::vector<int> hmap(256);
    for (int i = 0; i < 256; ++i) hmap[i] = 132 + i;
    add(L.pts[5], 256, 256, 256, hmap);
    add(L.pts[5], 256, 256, 144, pe, 1);  // wait for the re-filled operand, accumulate
  }
  add(L.pts[6], 256, 256, 256, identity_map(256, 256));
  add(L.pts[7], 256, 256, 256, identity_map(256, 256));
  add(L.coeff, 3 * n->nb, 32, 256, identity_map(256, 256));
  upload(img, tab, cur, left, &n->motion, st, &rc);
  return rc;
}

int launch_motion_fused(const dyn_net* n, MotionFusedArgs& a, cudaStream_t st) {
  a.producers = producer_lanes();
  if (!n->motion.img) return fail(DYN_E_INVALID, "motion net has no fused images");
  a.wimg = n->motion.img; a.chunks = n->motion.tab; a.nchunks = n->motion.nchunks;
  a.params = n->params;
  for (int i = 0; i < 8; ++i) a.o_bias[i] = n->ml.pts[i].b;
  a.o_bias[8] = n->ml.coeff.b;
  a.ncoef = 3 * n->nb;
  ProfScope prof(PROF_MOTION, st);
  return launch_chain(motion_fused_kernel, a, a.N, st);
}

}  // namespace dyn
