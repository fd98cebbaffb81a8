// Host-side launch of the fused per-(point, view) stage of the two aggregation networks: argument
// block, then the sub-round pipelined twin-warp kernel (view_twin3.cu).
//
// Reference semantics: ibrnet/projection.py:103-176, ibrnet/mlp_network.py:236-284
// (dynamic) and :423-497 (static).
#include <stdlib.h>

#include "fused_engine.cuh"
#include "geometry.cuh"
#include "nets.cuh"

namespace dyn {

// dyn_debug_set_view_kernel: -1 = the library's kernel.  Any other id (those of the removed comparison
// variants in particular) makes every fused per-view launch fail, so a measurement that asks for a variant
// cannot silently time the default under its name.
static int g_view_kernel = -1;
void set_view_kernel(int which) { g_view_kernel = which; }

// dyn_debug_set_view_kernel ids 0..2 (bench.py --view-kernel twin|quad|pipe)
static const char* const kRemovedViewKernels[3] = {"round-1 twin-warp kernel ('twin')", "quad-schedule kernel ('quad')",
                                                   "twin3 without elected arrive ('pipe')"};

int producer_lanes() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DYN_PRODUCERS");
    v = (e != nullptr && e[0] == '2') ? 2 : 1;  // two lanes of ONE warp do not help (divergence): r02_view_kernels.md
  }
  return v;
}

int launch_view_fused(const dyn_net* n, ViewFusedArgs& a, int V, cudaStream_t st) {
  if (g_view_kernel >= 0 && g_view_kernel < 3)
    return fail(DYN_E_INVALID, "per-view kernel variant %d, the %s, was removed; dyn_debug_set_view_kernel(-1) "
                "selects the library's kernel", g_view_kernel, kRemovedViewKernels[g_view_kernel]);
  if (g_view_kernel != -1)
    return fail(DYN_E_INVALID, "no per-view kernel variant %d; dyn_debug_set_view_kernel(-1) selects the library's "
                "kernel", g_view_kernel);
  if (V > 16) return fail(DYN_E_INVALID, "fused per-view kernel supports V <= 16 (got %d)", V);
  a.params = n->params;
  a.producers = producer_lanes();
  const bool st_net = n->kind == DYN_NET_STATIC;
  if (st_net) {
    const StaticLayout& L = n->sl;
    a.o_b1 = L.ray_dir0.b; a.o_b2 = L.ray_dir2.b; a.o_b3 = L.base0.b; a.o_b4 = L.base2.b;
    a.o_b5 = L.vis0.b; a.o_b6 = L.vis2.b; a.o_w6 = L.vis2.w; a.o_b7 = L.vis2_0.b;
    a.o_w8 = L.vis2_2.w; a.o_b8 = L.vis2_2.b; a.o_s = L.s;
    a.anti_alias = n->anti_alias; a.mask_rgb = n->mask_rgb;
  } else {
    const DynamicLayout& L = n->dl;
    a.o_b1 = 0; a.o_b2 = 0; a.o_b3 = L.base0.b; a.o_b4 = L.base2.b;
    a.o_b5 = L.vis0.b; a.o_b6 = L.vis2.b; a.o_w6 = L.vis2.w; a.o_b7 = L.vis2_0.b;
    a.o_w8 = L.vis2_2.w; a.o_b8 = L.vis2_2.b; a.o_s = -1;
    a.anti_alias = 0; a.mask_rgb = 0;
  }
  return launch_view_twin3(n, a, V, st);
}

}  // namespace dyn
