// libmeshnav_b200.so -- C ABI (include/meshnav_b200.h) over the sm_100a kernels.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false -std=c++17
//             -Xcompiler -fPIC -shared -o libmeshnav_b200.so meshnav.cu
#include <cuda_runtime.h>

#include <algorithm>
#include <functional>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/meshnav_b200.h"
#include "band_engine.cuh"
#include "problems.cuh"
#include "topology.hpp"

using namespace mnb;

#include "launch.cuh"
#include "kernels_maps.cuh"
#include "kernels_wavefront.cuh"
#include "dijkstra_batch.cuh"
#include "kernels_layers.cuh"
#include "kernels_field.cuh"
#include "kernels_updates.cuh"
#include "kernels_raycast.cuh"

// ============================================================================
// host side
// ============================================================================
struct mnb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int ptr_mode = MNB_PTR_HOST;
  int sm_count = 0;
  // mesh
  uint32_t V = 0, F = 0, E = 0;
  size_t NC = 0, NA = 0;
  HostTopology topo;
  float* d_pos = nullptr; uint32_t* d_faces = nullptr; uint32_t* d_edges = nullptr;
  uint32_t* d_cor_ptr = nullptr; int4* d_cor_idx = nullptr; uint4* d_cor_eid = nullptr; uint32_t* d_face_cor = nullptr;
  float4* d_cor_w = nullptr; float4* d_cor_wd = nullptr;
  int4* d_ell_idx = nullptr; uint4* d_ell_eid = nullptr; float4* d_ell_w = nullptr; float4* d_ell_wd = nullptr; double4* d_ell_geo = nullptr;
  uint32_t* d_adj_ptr = nullptr; uint32_t* d_adj_nbr = nullptr; uint32_t* d_adj_eid = nullptr; uint2* d_adj_nw = nullptr; uint4* d_ell_adj = nullptr;
  float* d_edge_dist = nullptr; float* d_edge_w = nullptr; float* d_cost = nullptr; uint8_t* d_invalid = nullptr;
  bool has_invalid = false, costs_set = false;
  bool adj_dirty = true;       // the Dijkstra planner's weight tables (adj_nw, ell_adj) are rebuilt on its first call after new weights
  // workspace
  uint32_t ws_groups = 0;
  WaveWorkspace ws{};
  unsigned int* d_next_query = nullptr;
  int* h_cancel = nullptr; int* d_cancel = nullptr;
  // scratch outputs for host-pointer mode
  float* d_out_dist = nullptr; size_t out_dist_cap = 0;
  uint32_t* d_out_pred = nullptr; float* d_out_dir = nullptr; int32_t* d_out_cut = nullptr;
  uint32_t* d_seed_faces = nullptr; float* d_seed_pos = nullptr; uint32_t seed_cap = 0;
  float* d_face_normals = nullptr; float* d_vertex_normals = nullptr; uint8_t* d_border = nullptr;
  float* d_layer_costs = nullptr; float* d_layer_combined = nullptr; uint8_t* d_layer_mask = nullptr; float* d_clearance = nullptr;
  float4* d_pos4 = nullptr; float4* d_vn4 = nullptr; uint32_t* d_nbr8 = nullptr;     // packed copies for k_layers<true>
  unsigned int* d_overflow = nullptr;
  // device-resident result of the last single CVP plan (for mnb_cvp_backtrack)
  const uint32_t* last_pred = nullptr; const float* last_dir = nullptr; const int32_t* last_cut = nullptr;
  uint32_t last_seed_face = 0; float last_seed_pos[3] = {0, 0, 0}; bool last_valid = false;
  float* d_path_pos = nullptr; uint32_t* d_path_face = nullptr; int32_t* d_bt_result = nullptr; uint32_t path_cap = 0;
  // scratch of mnb_dijkstra_batch (dijkstra_batch.cuh): its own, so that a batch leaves the wavefront workspace and the
  // device-resident result of the last mnb_cvp alone
  uint32_t* d_djb_scratch = nullptr; GroupCtl* d_djb_ctl = nullptr; uint32_t djb_groups = 0;
  uint32_t* d_djb_seeds = nullptr; uint32_t djb_seed_cap = 0; uint32_t* d_djb_pred = nullptr; size_t djb_pred_cap = 0;
  uint32_t* d_lethals = nullptr; uint32_t lethal_cap = 0; uint8_t* d_infl_invalid = nullptr; float* d_out_cost = nullptr;
  // repulsive vector field of the last inflation (InflationLayer::vector_map_ / distances_)
  bool infl_labels_valid = false, infl_had_invalid = false, infl_field_valid = false, repulsive_on = false;
  mnb_inflation_params infl_params{}; uint64_t infl_rounds = 0;
  float* d_infl_vec = nullptr; float* d_infl_dist = nullptr; int4* d_infl_src = nullptr; unsigned int* d_infl_flag = nullptr;
  // incremental updates
  float* d_prev_risk = nullptr; bool prev_risk_valid = false;     // riskiness map of the previous inflation (NaN = no entry)
  uint32_t* d_upd_ids = nullptr; float* d_upd_costs = nullptr; size_t upd_cap = 0; size_t upd_cost_cap = 0;
  uint32_t* d_upd_stamp = nullptr; uint32_t upd_call = 0;      // change-set membership stamps of mnb_update_vertex_costs
  uint32_t* d_changed = nullptr; unsigned int* d_tile_count = nullptr; unsigned int* d_total = nullptr;
  // tuning
  float delta = 0.3f; int cluster = -1 /* -1: whole-grid cooperative kernel for single plans */; int batch_cluster = 0 /* 0: chosen per call from the goal count */; int threads = 512;
  int grid_blocks_per_sm = 0;
  int infl_skip_clean = 1;     // clean-candidate skip of the inflation wave (MNB_INFL_SKIP=0 turns it off)
  int layers_smem = 5;         // neighbourhood walk of k_layers: 0 thread-local seen-set, 1 shared-memory seen-set, 2-4 prefetching walk (64 / 128 / 32
                               // threads per CTA), 5-7 the same with the 16-bit seen-set (64 / 128 / 256), 8-9 its low-register builds.  5 M vertices on
                               // the B200: 8.4 / - / 6.9 / ... / 5.1 ms for modes 0 / 2 / 5.  Chosen per mesh by mnb_set_mesh unless fixed by the caller.
  bool layers_explicit = false;
  int skip_clean = 0;          // clean-candidate stamps of the generic 8-lane CVP loop: measured slower on the B200 (35.8 vs 31.5 ms), its kernel
                               // instantiations are no longer built; the flag only reaches the legacy per-cluster kernel args.  The batch engine
                               // and the inflation wave carry their own (exact) rule.
  int sweeps = -1;             // in-round sweeps of the whole-grid single-plan kernel; -1 = derived from the band width
  float grid_delta = 1.8f;     // band width of the whole-grid single-plan kernel (wide band + in-round sweeps)
  float dijkstra_grid_delta = 3.0f;
  // The band widths above are potentials, i.e. multiples of the edge weights: unless the caller fixed them (mnb_set_tuning
  // with band_delta > 0) they follow the mean finite edge weight w of the installed weights -- 2.5 w for batches, 20 w for a
  // single CVP plan, 25 w for a single Dijkstra plan, less on maps above ~12 M vertices (install_weights); one dependency hop is
  // ~1.35 w (the in-round sweeps are counted in hops).  On the 0.1 m bench meshes (w = 0.118) that is 0.3 / 2.4 / 3.0 m, the values
  // the kernels were tuned with.
  bool delta_explicit = false; float w_mean = 0.0f; double* d_wsum = nullptr;
  int grid_engine = 0;         // experiment: 1 = full-field single plans run the lean batch round loop on the whole grid (k_cvp_batch<0>)
  float grid2_delta_w = 2.5f;  //             its band width in mean edge weights
  // ray caster over the faces (kernels_raycast.cuh; built on first use) + state of the obstacle layer
  RayBvh bvh{}; bool bvh_valid = false; unsigned int* d_ray_overflow = nullptr;
  float* d_ray_in = nullptr; size_t ray_in_cap = 0; float* d_ray_out = nullptr; size_t ray_out_cap = 0;
  uint8_t* d_obst_now = nullptr; uint8_t* d_obst_mask = nullptr; float* d_obst_member = nullptr; float* d_obst_member_chg = nullptr;
  uint32_t* d_obst_list = nullptr;
  mnb_stats stats{};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

#define CK(call)                                                                   \
  do {                                                                             \
    cudaError_t e_ = (call);                                                       \
    if (e_ != cudaSuccess) {                                                       \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
      return MNB_E_CUDA;                                                           \
    }                                                                              \
  } while (0)

template <class T>
static cudaError_t dalloc(T** p, size_t n) { return cudaMalloc((void**)p, n * sizeof(T) > 0 ? n * sizeof(T) : 1); }
template <class T>
static void dfree(T*& p) { if (p) cudaFree(p); p = nullptr; }

static void free_raycaster(mnb_ctx* c);
static void free_mesh(mnb_ctx* c) {
  free_raycaster(c);
  dfree(c->d_pos); dfree(c->d_faces); dfree(c->d_edges); dfree(c->d_cor_ptr); dfree(c->d_cor_idx); dfree(c->d_cor_eid); dfree(c->d_face_cor);
  dfree(c->d_cor_w); dfree(c->d_cor_wd); dfree(c->d_ell_idx); dfree(c->d_ell_eid); dfree(c->d_ell_w); dfree(c->d_ell_wd); dfree(c->d_ell_geo); dfree(c->d_adj_ptr); dfree(c->d_adj_nbr); dfree(c->d_adj_eid); dfree(c->d_adj_nw); dfree(c->d_ell_adj);
  dfree(c->d_edge_dist); dfree(c->d_edge_w); dfree(c->d_cost); dfree(c->d_invalid); dfree(c->d_wsum);
  dfree(c->ws.state); dfree(c->ws.ext); dfree(c->ws.pool); dfree(c->ws.skipw); dfree(c->ws.root); dfree(c->ws.last_eval); dfree(c->ws.dirty); dfree(c->ws.excl); dfree(c->ws.chg); dfree(c->ws.ver); dfree(c->ws.mark); dfree(c->ws.list0); dfree(c->ws.list1); dfree(c->ws.ctl);
  c->ws_groups = 0;
  dfree(c->d_out_dist); c->out_dist_cap = 0; dfree(c->d_out_pred); dfree(c->d_out_dir); dfree(c->d_out_cut);
  dfree(c->d_infl_invalid); dfree(c->d_out_cost);
  dfree(c->d_infl_vec); dfree(c->d_infl_dist); dfree(c->d_infl_src); dfree(c->d_infl_flag);
  c->infl_labels_valid = false; c->infl_field_valid = false; c->repulsive_on = false;
  dfree(c->d_prev_risk); c->prev_risk_valid = false; dfree(c->d_upd_ids); dfree(c->d_upd_costs); c->upd_cap = 0; c->upd_cost_cap = 0; dfree(c->d_upd_stamp); c->upd_call = 0;
  dfree(c->d_changed); dfree(c->d_tile_count); dfree(c->d_total);
  dfree(c->d_djb_scratch); dfree(c->d_djb_ctl); c->djb_groups = 0; dfree(c->d_djb_pred); c->djb_pred_cap = 0;
  dfree(c->d_path_pos); dfree(c->d_path_face); dfree(c->d_bt_result); c->path_cap = 0; c->last_valid = false;
  dfree(c->d_face_normals); dfree(c->d_vertex_normals); dfree(c->d_border); dfree(c->d_layer_costs); dfree(c->d_layer_combined);
  dfree(c->d_layer_mask); dfree(c->d_clearance); dfree(c->d_overflow); dfree(c->d_pos4); dfree(c->d_vn4); dfree(c->d_nbr8);
  c->costs_set = false;
}

static int32_t ensure_workspace(mnb_ctx* ctx, uint32_t groups) {
  if (groups <= ctx->ws_groups) return MNB_OK;
  dfree(ctx->ws.state); dfree(ctx->ws.ext); dfree(ctx->ws.pool); dfree(ctx->ws.skipw); dfree(ctx->ws.root); dfree(ctx->ws.last_eval); dfree(ctx->ws.dirty); dfree(ctx->ws.excl); dfree(ctx->ws.chg); dfree(ctx->ws.ver); dfree(ctx->ws.mark); dfree(ctx->ws.list0); dfree(ctx->ws.list1); dfree(ctx->ws.ctl);
  ctx->ws_groups = 0;
  const size_t n = (size_t)groups * ctx->V;
  CK(dalloc(&ctx->ws.state, n)); CK(dalloc(&ctx->ws.ext, n)); CK(dalloc(&ctx->ws.skipw, n)); CK(dalloc(&ctx->ws.root, n)); CK(dalloc(&ctx->ws.last_eval, n)); CK(dalloc(&ctx->ws.dirty, n)); CK(dalloc(&ctx->ws.excl, n)); CK(dalloc(&ctx->ws.chg, n)); CK(dalloc(&ctx->ws.ver, (size_t)ctx->V)); CK(dalloc(&ctx->ws.mark, n)); CK(dalloc(&ctx->ws.list0, n)); CK(dalloc(&ctx->ws.list1, n));
  // level pool (band_engine.cuh): pop times with more than 3 cascade levels keep their tails here; 2 words per vertex
  // hold the deepest flooded pockets randomised testing has produced with room to spare; exhaustion is reported
  ctx->ws.pool_cap = (uint32_t)std::min<size_t>(std::max<size_t>(65536, 2 * (size_t)ctx->V), 0x7fffffffu);
  CK(dalloc(&ctx->ws.pool, (size_t)groups * ctx->ws.pool_cap));
  CK(dalloc(&ctx->ws.ctl, groups));
  ctx->ws_groups = groups;
  return MNB_OK;
}

// Runs the body of a C-ABI entry point: std::bad_alloc (the host tables of a 50M-vertex map are tens of GB) becomes
// MNB_E_NOMEM, anything else MNB_E_STATE; a failed mnb_set_mesh frees what it had built so that later calls see an empty
// context instead of a half-built one.
template <class F>
static int32_t guarded(mnb_ctx* ctx, F body) {
  try {
    return body();
  } catch (const std::bad_alloc&) {
    if (ctx) ctx->err = "out of host memory";
    return MNB_E_NOMEM;
  } catch (const std::exception& ex) {
    if (ctx) ctx->err = ex.what();
    return MNB_E_STATE;
  } catch (...) {
    if (ctx) ctx->err = "unknown exception";
    return MNB_E_STATE;
  }
}

extern "C" {

int32_t mnb_create(int32_t device, mnb_ctx** out_ctx) {
  if (!out_ctx) return MNB_E_ARG;
  *out_ctx = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return MNB_E_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MNB_E_CUDA;
  if (prop.major < 10) return MNB_E_CUDA;   // sm_100a only; no fallback path exists
  if (cudaSetDevice(device) != cudaSuccess) return MNB_E_CUDA;
  mnb_ctx* c = new mnb_ctx();
  c->device = device; c->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("MNB_INFL_SKIP")) c->infl_skip_clean = atoi(e) != 0;                                 // experiment knob
  if (const char* e = getenv("MNB_LAYERS_SMEM")) { c->layers_smem = atoi(e); c->layers_explicit = true; }                                   // experiment knob
  if (const char* e = getenv("MNB_SKIP_CLEAN")) c->skip_clean = atoi(e) != 0;                                     // experiment knob
  if (const char* e = getenv("MNB_GRID_ENGINE")) c->grid_engine = atoi(e);                                     // experiment knob
  if (const char* e = getenv("MNB_GRID2_DELTA_W")) { const float k = (float)atof(e); if (k > 0) c->grid2_delta_w = k; }
  if (const char* e = getenv("MNB_SWEEPS")) { const int k = atoi(e); if (k >= -1 && k <= 64) c->sweeps = k; }   // experiment knob
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return MNB_E_CUDA; }
  cudaEventCreate(&c->ev0); cudaEventCreate(&c->ev1);
  cudaMalloc((void**)&c->d_next_query, sizeof(unsigned int));
  if (cudaHostAlloc((void**)&c->h_cancel, sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
    *c->h_cancel = 0;
    cudaHostGetDevicePointer((void**)&c->d_cancel, c->h_cancel, 0);
  }
  *out_ctx = c;
  return MNB_OK;
}

void mnb_destroy(mnb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  free_mesh(ctx);
  dfree(ctx->d_next_query); dfree(ctx->d_seed_faces); dfree(ctx->d_seed_pos); dfree(ctx->d_lethals); dfree(ctx->d_djb_seeds);
  if (ctx->h_cancel) cudaFreeHost(ctx->h_cancel);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* mnb_last_error(mnb_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
int32_t mnb_set_pointer_mode(mnb_ctx* ctx, int32_t mode) {
  if (!ctx || (mode != MNB_PTR_HOST && mode != MNB_PTR_DEVICE)) return MNB_E_ARG;
  ctx->ptr_mode = mode; return MNB_OK;
}
void* mnb_stream(mnb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
uint32_t mnb_num_vertices(mnb_ctx* ctx) { return ctx ? ctx->V : 0; }
uint32_t mnb_num_faces(mnb_ctx* ctx) { return ctx ? ctx->F : 0; }
uint32_t mnb_num_edges(mnb_ctx* ctx) { return ctx ? ctx->E : 0; }

int32_t mnb_set_tuning(mnb_ctx* ctx, float band_delta, int32_t cluster_size, int32_t threads_per_cta) {
  if (!ctx) return MNB_E_ARG;
  if (band_delta > 0) { ctx->delta = band_delta; ctx->grid_delta = band_delta; ctx->dijkstra_grid_delta = band_delta; ctx->delta_explicit = true; }
  if (cluster_size == 1 || cluster_size == 2 || cluster_size == 4 || cluster_size == 8 || cluster_size == 16) {
    ctx->cluster = cluster_size;
    ctx->batch_cluster = cluster_size > 8 ? 8 : cluster_size;
  } else if (cluster_size == -1) {
    ctx->cluster = -1;        // single plans on the whole grid (cooperative launch); batches keep their cluster size
  } else if (cluster_size != 0) return MNB_E_ARG;
  if (threads_per_cta == 128 || threads_per_cta == 256 || threads_per_cta == 512) { ctx->threads = threads_per_cta; ctx->grid_blocks_per_sm = 0; }
  else if (threads_per_cta != 0) return MNB_E_ARG;
  return MNB_OK;
}

int32_t mnb_get_stats(mnb_ctx* ctx, mnb_stats* out) {
  if (!ctx || !out) return MNB_E_ARG;
  *out = ctx->stats; return MNB_OK;
}

static int32_t impl_set_mesh(mnb_ctx* ctx, uint32_t V, uint32_t F, const float* pos, const uint32_t* faces,
                     const uint32_t* edges, uint32_t E) {
  if (!ctx || !pos || !faces || V == 0 || F == 0) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  free_mesh(ctx);
  try {
    ctx->topo.build(V, F, faces, edges, E);
  } catch (const std::exception& ex) {
    ctx->err = ex.what();
    return MNB_E_ARG;
  }
  HostTopology& T = ctx->topo;
  if (!ctx->layers_explicit) {
    // the compact seen-set of the layer walk (walk_pf16) holds ids within +-32767 of the centre's: a neighbourhood reaches a
    // few edges out, so it pays when edges connect nearby ids (scan / Morton numbering); otherwise the 32-bit form
    uint32_t maxd = 0;
    for (size_t e = 0; e < (size_t)T.E; ++e) { const uint32_t a = T.edges[2 * e], b = T.edges[2 * e + 1]; maxd = std::max(maxd, a > b ? a - b : b - a); }
    ctx->layers_smem = (maxd <= 8000u) ? 5 : 2;
  }
  ctx->V = V; ctx->F = F; ctx->E = T.E; ctx->NC = T.cor_v1.size(); ctx->NA = T.vadj_nbr.size();
  const size_t NC = ctx->NC, NA = ctx->NA;
  CK(dalloc(&ctx->d_pos, 3 * (size_t)V)); CK(dalloc(&ctx->d_faces, 3 * (size_t)F)); CK(dalloc(&ctx->d_edges, 2 * (size_t)T.E));
  CK(dalloc(&ctx->d_cor_ptr, (size_t)V + 1)); CK(dalloc(&ctx->d_cor_idx, NC)); CK(dalloc(&ctx->d_cor_eid, NC));
  CK(dalloc(&ctx->d_cor_w, NC)); CK(dalloc(&ctx->d_cor_wd, NC));
  CK(dalloc(&ctx->d_adj_ptr, (size_t)V + 1)); CK(dalloc(&ctx->d_adj_nbr, NA)); CK(dalloc(&ctx->d_adj_eid, NA)); CK(dalloc(&ctx->d_adj_nw, NA)); CK(dalloc(&ctx->d_ell_adj, (size_t)V * ELL_W));
  CK(dalloc(&ctx->d_edge_dist, (size_t)T.E)); CK(dalloc(&ctx->d_edge_w, (size_t)T.E)); CK(dalloc(&ctx->d_cost, (size_t)V));
  CK(dalloc(&ctx->d_invalid, (size_t)V));
  CK(cudaMemcpyAsync(ctx->d_pos, pos, sizeof(float) * 3 * (size_t)V, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_faces, faces, sizeof(uint32_t) * 3 * (size_t)F, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_edges, T.edges.data(), sizeof(uint32_t) * 2 * (size_t)T.E, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_cor_ptr, T.vcor_ptr.data(), sizeof(uint32_t) * ((size_t)V + 1), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_adj_ptr, T.vadj_ptr.data(), sizeof(uint32_t) * ((size_t)V + 1), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_adj_nbr, T.vadj_nbr.data(), sizeof(uint32_t) * NA, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_adj_eid, T.vadj_eid.data(), sizeof(uint32_t) * NA, cudaMemcpyHostToDevice, ctx->stream));
  {
    std::vector<int4> idx(NC); std::vector<uint4> eid(NC);
    for (size_t k = 0; k < NC; ++k) {
      idx[k] = make_int4((int)T.cor_v1[k], (int)T.cor_v2[k], (int)T.cor_face[k], (int)T.cor_side[k]);   // .w: edge-side bits (topology.hpp)
      eid[k] = make_uint4(T.cor_ec[k], T.cor_eb[k], T.cor_ea[k], 0);
    }
    CK(cudaMemcpyAsync(ctx->d_cor_idx, idx.data(), sizeof(int4) * NC, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_cor_eid, eid.data(), sizeof(uint4) * NC, cudaMemcpyHostToDevice, ctx->stream));
    CK(dalloc(&ctx->d_face_cor, 3 * (size_t)F));
    CK(cudaMemcpyAsync(ctx->d_face_cor, T.face_cor.data(), sizeof(uint32_t) * 3 * (size_t)F, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // ELL rows: 8 slots per vertex (one 128-byte line), slot 0 carries the degree in .w
    const size_t NE = (size_t)V * ELL_W;
    std::vector<int4> eidx(NE, make_int4(ELL_EMPTY, ELL_EMPTY, -1, 0)); std::vector<uint4> eeid(NE, make_uint4(0, 0, 0, 0));
    for (uint32_t v = 0; v < V; ++v) {
      const uint32_t kb = T.vcor_ptr[v], ke = T.vcor_ptr[v + 1];
      for (uint32_t k = kb; k < ke && k - kb < ELL_W; ++k) { eidx[(size_t)v * ELL_W + (k - kb)] = idx[k]; eeid[(size_t)v * ELL_W + (k - kb)] = eid[k]; }
      eidx[(size_t)v * ELL_W].w = (int)(ke - kb);
    }
    CK(dalloc(&ctx->d_ell_idx, NE)); CK(dalloc(&ctx->d_ell_eid, NE)); CK(dalloc(&ctx->d_ell_w, NE)); CK(dalloc(&ctx->d_ell_wd, NE));
    CK(dalloc(&ctx->d_ell_geo, NE));
    CK(cudaMemcpyAsync(ctx->d_ell_idx, eidx.data(), sizeof(int4) * NE, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_ell_eid, eeid.data(), sizeof(uint4) * NE, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  // the host copies of the big per-corner arrays are no longer needed
  std::vector<uint32_t>().swap(T.cor_v1); std::vector<uint32_t>().swap(T.cor_v2); std::vector<uint32_t>().swap(T.cor_face);
  std::vector<uint32_t>().swap(T.cor_ec); std::vector<uint32_t>().swap(T.cor_eb); std::vector<uint32_t>().swap(T.cor_ea);
  std::vector<uint8_t>().swap(T.cor_side);
  std::vector<uint32_t>().swap(T.vadj_nbr); std::vector<uint32_t>().swap(T.vadj_eid); std::vector<uint32_t>().swap(T.face_edges);
  CK(dalloc(&ctx->d_face_normals, 3 * (size_t)F)); CK(dalloc(&ctx->d_vertex_normals, 3 * (size_t)V)); CK(dalloc(&ctx->d_border, (size_t)V));
  CK(cudaMemcpyAsync(ctx->d_border, T.border.data(), (size_t)V, cudaMemcpyHostToDevice, ctx->stream));
  MNB_LAUNCH(k_face_normals, (F + 255) / 256, 256, 0, ctx->stream, ctx->d_pos, ctx->d_faces, F, ctx->d_face_normals);
  MNB_LAUNCH(k_vertex_normals, (V + 255) / 256, 256, 0, ctx->stream, ctx->d_cor_ptr, ctx->d_cor_idx, ctx->d_face_normals, V, ctx->d_vertex_normals);
  MNB_LAUNCH(k_edge_dist, (T.E + 255) / 256, 256, 0, ctx->stream, ctx->d_pos, ctx->d_edges, T.E, ctx->d_edge_dist);
  MNB_LAUNCH(k_gather_corner_w, (unsigned)((NC + 255) / 256), 256, 0, ctx->stream, ctx->d_cor_eid, ctx->d_edge_dist, NC, ctx->d_cor_wd);
  MNB_LAUNCH(k_gather_corner_w, (unsigned)(((size_t)V * ELL_W + 255) / 256), 256, 0, ctx->stream, ctx->d_ell_eid, ctx->d_edge_dist, (size_t)V * ELL_W, ctx->d_ell_wd);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

int32_t mnb_get_edges(mnb_ctx* ctx, uint32_t* out_edges) {
  if (!ctx || !out_edges || !ctx->V) return MNB_E_ARG;
  std::memcpy(out_edges, ctx->topo.edges.data(), sizeof(uint32_t) * 2 * (size_t)ctx->E);
  return MNB_OK;
}

static cudaMemcpyKind in_kind(mnb_ctx* c) { return c->ptr_mode == MNB_PTR_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice; }
static cudaMemcpyKind out_kind(mnb_ctx* c) { return c->ptr_mode == MNB_PTR_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice; }

int32_t mnb_get_edge_distances(mnb_ctx* ctx, float* out) {
  if (!ctx || !out || !ctx->V) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(out, ctx->d_edge_dist, sizeof(float) * (size_t)ctx->E, out_kind(ctx), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

static int32_t install_weights(mnb_ctx* ctx) {
  MNB_LAUNCH(k_gather_corner_w, (unsigned)((ctx->NC + 255) / 256), 256, 0, ctx->stream, ctx->d_cor_eid, ctx->d_edge_w, ctx->NC, ctx->d_cor_w);
  MNB_LAUNCH(k_gather_corner_w, (unsigned)(((size_t)ctx->V * ELL_W + 255) / 256), 256, 0, ctx->stream, ctx->d_ell_eid, ctx->d_edge_w, (size_t)ctx->V * ELL_W, ctx->d_ell_w);
  MNB_LAUNCH(k_corner_geo, (unsigned)(((size_t)ctx->V * ELL_W + 255) / 256), 256, 0, ctx->stream, ctx->d_ell_w, (size_t)ctx->V * ELL_W, ctx->d_ell_geo);
  ctx->adj_dirty = true;        // adjacency form of the weights: only the Dijkstra planner reads it (ensure_adj_tables)
  CK(cudaGetLastError());
  // scale of the potentials: mean finite edge weight (see mnb_ctx::delta_explicit)
  if (!ctx->d_wsum) CK(dalloc(&ctx->d_wsum, 2));
  CK(cudaMemsetAsync(ctx->d_wsum, 0, 2 * sizeof(double), ctx->stream));
  MNB_LAUNCH(k_weight_scale, 296, 256, 0, ctx->stream, (const float*)ctx->d_edge_w, ctx->E, ctx->d_wsum);
  CK(cudaGetLastError());
  double hs[2] = {0.0, 0.0};
  CK(cudaMemcpyAsync(hs, ctx->d_wsum, sizeof(hs), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->w_mean = hs[1] > 0 ? (float)(hs[0] / hs[1]) : 0.0f;
  if (!ctx->delta_explicit && ctx->w_mean > 0) {
    // Single plans: the band should hold about as many candidates as the grid has sweep slots (SM count x Stage::SW_CAP);
    // beyond that the in-round sweeps cannot follow and the band's rows fall out of the L2.  A front is ~3 sqrt(V) vertices
    // long on a compact map and a hop is ~1.35 w deep.  5 M vertices: 20 w / 25 w (the values the kernels were tuned with);
    // 50 M: 9.6 w -- measured there: CVP 342 -> 232 ms, Dijkstra 178 -> 98 ms against the fixed 20 w / 25 w.
    const float slots = (float)ctx->sm_count * (float)Stage::SW_CAP;
    const float hops = slots / (3.0f * sqrtf((float)ctx->V));
    const float k = fmaxf(4.0f, 1.35f * hops);
    ctx->delta = 2.5f * ctx->w_mean;
    ctx->grid_delta = fminf(20.0f, k) * ctx->w_mean;
    ctx->dijkstra_grid_delta = fminf(25.0f, k) * ctx->w_mean;
  }
  ctx->costs_set = true;
  return MNB_OK;
}

// the vertex->neighbour form of the installed weights (CSR {neighbour, weight} + the 8-slot ELL rows of k_dijkstra_grid)
static int32_t ensure_adj_tables(mnb_ctx* ctx) {
  if (!ctx->adj_dirty) return MNB_OK;
  MNB_LAUNCH(k_gather_adj_w, (unsigned)((ctx->NA + 255) / 256), 256, 0, ctx->stream, ctx->d_adj_nbr, ctx->d_adj_eid, ctx->d_edge_w, ctx->NA, ctx->d_adj_nw);
  MNB_LAUNCH(k_build_ell_adj, (unsigned)(((size_t)ctx->V * ELL_W + 255) / 256), 256, 0, ctx->stream, ctx->d_adj_ptr, ctx->d_adj_nw, ctx->V, ctx->d_ell_adj);
  CK(cudaGetLastError());
  ctx->adj_dirty = false;
  return MNB_OK;
}

static int32_t impl_compute_edge_weights(mnb_ctx* ctx, const float* vertex_costs, double edge_cost_factor, float* out_w) {
  if (!ctx || !vertex_costs || !ctx->V) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(ctx->d_cost, vertex_costs, sizeof(float) * (size_t)ctx->V, in_kind(ctx), ctx->stream));
  MNB_LAUNCH(k_edge_weights, (ctx->E + 255) / 256, 256, 0, ctx->stream, ctx->d_cost, ctx->d_edges, ctx->d_edge_dist, edge_cost_factor, ctx->E, ctx->d_edge_w);
  CK(cudaGetLastError());
  int32_t rc = install_weights(ctx);
  if (rc != MNB_OK) return rc;
  if (out_w) CK(cudaMemcpyAsync(out_w, ctx->d_edge_w, sizeof(float) * (size_t)ctx->E, out_kind(ctx), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

static int32_t impl_set_costs(mnb_ctx* ctx, const float* vertex_costs, const float* edge_weights, const uint8_t* invalid) {
  if (!ctx || !vertex_costs || !edge_weights || !ctx->V) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(ctx->d_cost, vertex_costs, sizeof(float) * (size_t)ctx->V, in_kind(ctx), ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_edge_w, edge_weights, sizeof(float) * (size_t)ctx->E, in_kind(ctx), ctx->stream));
  if (invalid) CK(cudaMemcpyAsync(ctx->d_invalid, invalid, (size_t)ctx->V, in_kind(ctx), ctx->stream));
  ctx->has_invalid = invalid != nullptr;
  int32_t rc = install_weights(ctx);
  if (rc != MNB_OK) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

int32_t mnb_cancel(mnb_ctx* ctx) {
  if (!ctx || !ctx->h_cancel) return MNB_E_ARG;
  *(volatile int*)ctx->h_cancel = 1;
  return MNB_OK;
}

}  // extern "C"


static RepulsiveField repulsive_field_of(mnb_ctx* ctx) {
  RepulsiveField L{};
  L.dist = ctx->d_infl_dist; L.vec = ctx->d_infl_vec;
  L.inscribed_radius = ctx->infl_params.inscribed_radius; L.inflation_radius = ctx->infl_params.inflation_radius;
  L.inscribed_radius_f = (float)ctx->infl_params.inscribed_radius;
  L.lethal_value = (float)ctx->infl_params.lethal_value; L.inscribed_value = (float)ctx->infl_params.inscribed_value;
  return L;
}

extern "C" {

static int32_t impl_inflation_vector_map(mnb_ctx* ctx, float* out_vectors) {
  if (!ctx || !ctx->V) return MNB_E_ARG;
  if (!ctx->infl_labels_valid) {
    ctx->err = "mnb_inflation_vector_map needs the labels of the last mnb_inflate / mnb_inflation_update: call it before the next planner call on this context";
    return MNB_E_STATE;
  }
  CK(cudaSetDevice(ctx->device));
  const size_t V = ctx->V;
  if (!ctx->d_infl_vec) { CK(dalloc(&ctx->d_infl_vec, 3 * V)); CK(dalloc(&ctx->d_infl_src, V)); CK(dalloc(&ctx->d_infl_flag, (size_t)2)); }
  InflVecArgs a{};
  a.V = ctx->V; a.pos = ctx->d_pos; a.faces = ctx->d_faces; a.cor_ptr = ctx->d_cor_ptr; a.cor_idx = ctx->d_cor_idx; a.cor_wd = ctx->d_cor_wd;
  a.cor_eid = ctx->d_cor_eid; a.adj_ptr = ctx->d_adj_ptr; a.adj_nbr = ctx->d_adj_nbr; a.invalid = ctx->infl_had_invalid ? ctx->d_infl_invalid : nullptr; a.ws = ctx->ws;
  a.max_distance = (float)ctx->infl_params.inflation_radius; a.vec = ctx->d_infl_vec; a.src = ctx->d_infl_src; a.flag = ctx->d_infl_flag;
  CK(cudaMemsetAsync(ctx->d_infl_flag, 0, 2 * sizeof(unsigned int), ctx->stream));
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  MNB_LAUNCH(k_infl_vec_lethal, (ctx->V + 127) / 128, 128, 0, ctx->stream, a);
  MNB_LAUNCH(k_infl_vec_sources, (ctx->V + 127) / 128, 128, 0, ctx->stream, a);
  CK(cudaGetLastError());
  unsigned launches = 2;
  // fixed point over the acyclic source relation: its depth is bounded by the number of rounds the wave took
  const unsigned max_sweeps = (unsigned)ctx->infl_rounds + 8u;
  unsigned int flag[2] = {1u, 0u};
  for (unsigned it = 0; it < max_sweeps && flag[0]; ++it, ++launches) {
    CK(cudaMemsetAsync(ctx->d_infl_flag, 0, sizeof(unsigned int), ctx->stream));
    MNB_LAUNCH(k_infl_vec_sweep, (ctx->V + 255) / 256, 256, 0, ctx->stream, a);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(flag, ctx->d_infl_flag, sizeof(flag), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (flag[1]) { ctx->err = "inflation vector field: a vertex has more than 24 faces with two lethal vertices"; return MNB_E_NOMEM; }
  if (flag[0]) { ctx->err = "inflation vector field did not reach its fixed point"; return MNB_E_STATE; }
  if (out_vectors) CK(cudaMemcpyAsync(out_vectors, ctx->d_infl_vec, sizeof(float) * 3 * V, out_kind(ctx), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const uint64_t wave_rounds = ctx->infl_rounds;
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = launches; ctx->stats.settled = ctx->V; ctx->stats.rounds = wave_rounds;
  ctx->infl_field_valid = true;
  return MNB_OK;
}

int32_t mnb_set_repulsive_field(mnb_ctx* ctx, int32_t enable) {
  if (!ctx) return MNB_E_ARG;
  if (enable && !ctx->infl_field_valid) { ctx->err = "mnb_set_repulsive_field needs mnb_inflation_vector_map first"; return MNB_E_STATE; }
  ctx->repulsive_on = enable != 0;
  return MNB_OK;
}

static int32_t impl_inflation_vector_at(mnb_ctx* ctx, uint32_t n, const uint32_t* faces_q, const float* bary, float* out) {
  if (!ctx || !ctx->V || !faces_q || !bary || !out || n == 0) return MNB_E_ARG;
  if (!ctx->infl_field_valid) { ctx->err = "mnb_inflation_vector_at needs mnb_inflation_vector_map first"; return MNB_E_STATE; }
  for (uint32_t i = 0; ctx->ptr_mode == MNB_PTR_HOST && i < n; ++i) if (faces_q[i] >= ctx->F) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  uint32_t* d_f = nullptr; float* d_b = nullptr; float* d_o = nullptr;
  if (!dev) {
    CK(dalloc(&d_f, (size_t)n)); CK(dalloc(&d_b, 3 * (size_t)n)); CK(dalloc(&d_o, 3 * (size_t)n));
    CK(cudaMemcpyAsync(d_f, faces_q, sizeof(uint32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_b, bary, sizeof(float) * 3 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  }
  MNB_LAUNCH(k_inflation_vector_at, (n + 127) / 128, 128, 0, ctx->stream, repulsive_field_of(ctx), (const uint32_t*)ctx->d_faces, n,
             dev ? faces_q : (const uint32_t*)d_f, dev ? bary : (const float*)d_b, dev ? out : d_o);
  CK(cudaGetLastError());
  if (!dev) CK(cudaMemcpyAsync(out, d_o, sizeof(float) * 3 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  dfree(d_f); dfree(d_b); dfree(d_o);
  return MNB_OK;
}

}  // extern "C"

template <class KArgs>
static cudaError_t launch_cluster(void (*kern)(const KArgs), const KArgs& args, int cs, unsigned blocks, int threads,
                                  cudaStream_t stream) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = cs > 1 ? 1 : 0;
  if (cs > 8) {
    cudaError_t e = cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
  }
  return cudaLaunchKernelEx(&cfg, kern, args);
}

// cooperative (grid-synchronising) launch of a kernel that takes one argument struct
template <class KArgs>
static cudaError_t launch_cooperative(void (*kern)(const KArgs), const KArgs& args, unsigned blocks, int threads, cudaStream_t stream) {
#ifdef MNB_EMU_ACTIVE
  (void)stream;
  return emu::launch(kern, blocks, (unsigned)threads, (size_t)0, 1u, true, args);
#else
  void* kargs[] = {(void*)&args};
  return cudaLaunchCooperativeKernel((const void*)kern, dim3(blocks), dim3(threads), kargs, 0, stream);
#endif
}

static int32_t launch_cvp(mnb_ctx* ctx, const CvpKernelArgs& a, int cs, unsigned groups) {
  cudaError_t e;
  const unsigned blocks = groups * cs;
  const int threads = MNB_CVP_THREADS;
  switch (cs) {
    case 1: e = launch_cluster(k_cvp<1, false>, a, 1, blocks, threads, ctx->stream); break;
    case 2: e = launch_cluster(k_cvp<2, false>, a, 2, blocks, threads, ctx->stream); break;     // (the skip variant is built for the two
    case 4: e = launch_cluster(k_cvp<4, false>, a, 4, blocks, threads, ctx->stream); break;     //  default configurations only: per-CTA batches
    case 8: e = launch_cluster(k_cvp<8, false>, a, 8, blocks, threads, ctx->stream); break;     //  and the whole-grid single plan)
    default: e = launch_cluster(k_cvp<16, false>, a, 16, blocks, threads, ctx->stream); break;
  }
  if (e != cudaSuccess) { ctx->err = std::string("cvp launch: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  return MNB_OK;
}

static int32_t finish_stats(mnb_ctx* ctx, unsigned groups, unsigned launches, const GroupCtl* ctl = nullptr) {
  std::vector<GroupCtl> h(groups);
  CK(cudaMemcpyAsync(h.data(), ctl ? ctl : ctx->ws.ctl, sizeof(GroupCtl) * groups, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->stats.rounds = 0; ctx->stats.recomputes = 0; ctx->stats.settled = 0;
  ctx->stats.skipped = 0; ctx->stats.deep_labels = 0; ctx->stats.pool_words = 0;
  for (auto& c : h) { ctx->stats.deep_labels += c.deep_labels; ctx->stats.pool_words = std::max<uint64_t>(ctx->stats.pool_words, c.pool_top); }
  for (auto& c : h) { ctx->stats.rounds += c.rounds; ctx->stats.recomputes += c.recomputes; ctx->stats.settled += c.settled; ctx->stats.skipped += c.skipped; }
  ctx->stats.kernel_launches = launches;
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1); ctx->stats.kernel_ms = ms;
  if (getenv("MNB_PHASE_TIMING")) for (auto& c : h) fprintf(stderr, "[mnb] rounds %llu: CTA0 cycles work %llu flush %llu sync %llu (per round %.0f / %.0f / %.0f) main-pass cycles %llu (unused %llu) chunk-candidates %llu | sweeps: dirty %llu polled %llu poll-cycles %llu eval-cycles %llu (%llu)\n", c.rounds, c.t_work, c.t_flush, c.t_sync, (double)c.t_work / (double)(c.rounds ? c.rounds : 1), (double)c.t_flush / (double)(c.rounds ? c.rounds : 1), (double)c.t_sync / (double)(c.rounds ? c.rounds : 1), c.t_ph[0], c.t_ph[1], c.t_ph[2], c.t_ph[3], c.t_ph[4], c.t_ph[5], c.t_ph[6], c.t_ph[7]);
  for (auto& c : h)
    if (c.watchdog) { ctx->err = "wavefront did not converge within the round watchdog"; return MNB_E_STATE; }
  for (auto& c : h)
    if (c.pool_overflow) { ctx->err = "level pool exhausted: the cascades of this map nest deeper than the workspace holds (result discarded)"; return MNB_E_NOMEM; }
  return MNB_OK;
}

static int32_t ensure_out(mnb_ctx* ctx, size_t n_dist, bool aux) {
  if (n_dist > ctx->out_dist_cap) { dfree(ctx->d_out_dist); CK(dalloc(&ctx->d_out_dist, n_dist)); ctx->out_dist_cap = n_dist; }
  if (aux && !ctx->d_out_pred) {
    CK(dalloc(&ctx->d_out_pred, (size_t)ctx->V)); CK(dalloc(&ctx->d_out_dir, (size_t)ctx->V)); CK(dalloc(&ctx->d_out_cut, (size_t)ctx->V));
  }
  return MNB_OK;
}

static int32_t ensure_seeds(mnb_ctx* ctx, uint32_t n) {
  if (n > ctx->seed_cap) {
    dfree(ctx->d_seed_faces); dfree(ctx->d_seed_pos);
    CK(dalloc(&ctx->d_seed_faces, (size_t)n)); CK(dalloc(&ctx->d_seed_pos, 3 * (size_t)n));
    ctx->seed_cap = n;
  }
  return MNB_OK;
}

static void fill_cvp_args(mnb_ctx* ctx, CvpKernelArgs& a) {
  a.V = ctx->V; a.pos = ctx->d_pos; a.faces = ctx->d_faces; a.cor_ptr = ctx->d_cor_ptr; a.cor_idx = ctx->d_cor_idx;
  a.cor_w = ctx->d_cor_w; a.ell_idx = ctx->d_ell_idx; a.ell_w = ctx->d_ell_w; a.ell_geo = ctx->d_ell_geo; a.cost = ctx->d_cost; a.invalid = ctx->has_invalid ? ctx->d_invalid : nullptr; a.ws = ctx->ws;
  a.seed_faces = ctx->d_seed_faces; a.seed_pos = ctx->d_seed_pos; a.delta = ctx->delta; a.next_query = ctx->d_next_query;
  a.cancel_flag = ctx->d_cancel; a.max_rounds = watchdog_rounds(ctx->V); a.sweeps = 0; a.skip_clean = ctx->skip_clean;
  a.hop = ctx->w_mean > 0 ? 1.35f * ctx->w_mean : 0.16f;
}

extern "C" {

static int32_t impl_cvp(mnb_ctx* ctx, uint32_t seed_face, const float seed_pos[3], int64_t robot_face, double cost_limit,
                double goal_dist_offset, float* out_dist, uint32_t* out_pred, float* out_direction, int32_t* out_cut) {
  if (!ctx || !seed_pos || !ctx->V) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "mnb_set_costs / mnb_compute_edge_weights not called"; return MNB_E_STATE; }
  if (seed_face >= ctx->F) return MNB_INVALID_START;
  if (robot_face >= (int64_t)ctx->F) return MNB_INVALID_GOAL;
  CK(cudaSetDevice(ctx->device));
  int32_t rc;
  if ((rc = ensure_workspace(ctx, 1)) != MNB_OK) return rc;
  if ((rc = ensure_seeds(ctx, 1)) != MNB_OK) return rc;
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  if ((rc = ensure_out(ctx, dev ? 0 : (size_t)ctx->V, true)) != MNB_OK) return rc;
  if (ctx->h_cancel) *ctx->h_cancel = 0;     // cvp:679 "reset cancel planning"
  ctx->infl_labels_valid = false;            // the wavefront workspace is shared with the inflation wave
  CK(cudaMemcpyAsync(ctx->d_seed_faces, &seed_face, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_seed_pos, seed_pos, 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->d_next_query, 0, sizeof(unsigned int), ctx->stream));
  CK(cudaMemsetAsync(ctx->ws.ctl, 0, sizeof(GroupCtl), ctx->stream));
  CvpKernelArgs a{};
  fill_cvp_args(ctx, a);
  a.n_queries = 1; a.robot_face = robot_face; a.cost_limit = cost_limit; a.goal_dist_offset = goal_dist_offset;
  a.sweeps = ctx->sweeps;
  a.out_dist = dev ? out_dist : ctx->d_out_dist;
  // aux outputs are always produced for a single plan (the outcome code needs predecessors_)
  a.out_pred = (dev && out_pred) ? out_pred : ctx->d_out_pred;
  a.out_dir = (dev && out_direction) ? out_direction : ctx->d_out_dir;
  a.out_cut = (dev && out_cut) ? out_cut : ctx->d_out_cut;
  if (dev && !out_dist) { if ((rc = ensure_out(ctx, (size_t)ctx->V, true)) != MNB_OK) return rc; a.out_dist = ctx->d_out_dist; }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  if (ctx->cluster == -1) {
    a.delta = ctx->grid_delta;
    if (ctx->grid_blocks_per_sm == 0) {
      int nb = 0;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_cvp_grid<false>, ctx->threads, 0));
      ctx->grid_blocks_per_sm = nb > MNB_GRID_MINBLOCKS ? MNB_GRID_MINBLOCKS : nb;
      if (nb <= 0) { ctx->err = "k_cvp_grid cannot be resident"; return MNB_E_CUDA; }
    }
    if (ctx->grid_engine == 1 && robot_face < 0) {
      int per_sm = 1;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cvp_batch<0>, MNB_BATCH_THREADS, 0));
      if (per_sm > MNB_BATCH_MINBLOCKS) per_sm = MNB_BATCH_MINBLOCKS;
      if (per_sm < 1) { ctx->err = "k_cvp_batch<0> cannot be resident"; return MNB_E_CUDA; }
      a.delta = ctx->grid2_delta_w * (ctx->w_mean > 0.0f ? ctx->w_mean : 0.12f);
      CK(launch_cooperative(k_cvp_batch<0>, a, (unsigned)(ctx->sm_count * per_sm), MNB_BATCH_THREADS, ctx->stream));
    } else
    CK(launch_cooperative(k_cvp_grid<false>, a, (unsigned)(ctx->sm_count * ctx->grid_blocks_per_sm), ctx->threads, ctx->stream));
  } else {
    if ((rc = launch_cvp(ctx, a, ctx->cluster, 1)) != MNB_OK) return rc;
  }
  MNB_LAUNCH(k_cvp_epilogue, (ctx->V + 255) / 256, 256, 0, ctx->stream, a, ctx->ws.ctl);
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    if (out_dist) CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_pred) CK(cudaMemcpyAsync(out_pred, a.out_pred, sizeof(uint32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_direction) CK(cudaMemcpyAsync(out_direction, a.out_dir, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_cut) CK(cudaMemcpyAsync(out_cut, a.out_cut, sizeof(int32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
  }
  // outcome (cvp:888-918)
  uint32_t rf[3] = {0, 0, 0}, rp[3] = {0, 0, 0};
  if (robot_face >= 0) {
    CK(cudaMemcpyAsync(rf, ctx->d_faces + 3 * (size_t)robot_face, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 3; ++k)
      CK(cudaMemcpyAsync(&rp[k], a.out_pred + rf[k], sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  }
  ctx->last_valid = false;
  if ((rc = finish_stats(ctx, 1, 2)) != MNB_OK) return rc;
  if (ctx->h_cancel && *ctx->h_cancel) return MNB_CANCELED;
  ctx->last_pred = a.out_pred; ctx->last_dir = a.out_dir; ctx->last_cut = a.out_cut; ctx->last_seed_face = seed_face;
  for (int k = 0; k < 3; ++k) ctx->last_seed_pos[k] = seed_pos[k];
  ctx->last_valid = true;
  if (robot_face >= 0) {
    bool any = false;
    for (int k = 0; k < 3; ++k) if (rp[k] != rf[k]) any = true;
    if (!any && (uint32_t)robot_face != seed_face) return MNB_NO_PATH_FOUND;
  }
  return MNB_SUCCESS;
}

static int32_t impl_cvp_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_faces, const float* seed_pos, double cost_limit,
                      float* out_dist) {
  if (!ctx || !seed_faces || !seed_pos || !out_dist || !ctx->V || n == 0) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "costs not set"; return MNB_E_STATE; }
  for (uint32_t i = 0; i < n; ++i) if (seed_faces[i] >= ctx->F) return MNB_INVALID_START;
  CK(cudaSetDevice(ctx->device));
  // resident CTAs per SM of the lean batch kernel (k_cvp_batch, batch_engine.cuh); MNB_BATCH_LEGACY=1 runs the generic
  // round loop (k_cvp) instead -- kept for A/B measurements
  static const bool legacy = getenv("MNB_BATCH_LEGACY") != nullptr;
  int per_sm = 1;
  if (legacy) { CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cvp<1, false>, MNB_CVP_THREADS, 0)); if (per_sm > 2) per_sm = 2; }
  else { CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cvp_batch<1>, MNB_BATCH_THREADS, 0)); if (per_sm > MNB_BATCH_MINBLOCKS) per_sm = MNB_BATCH_MINBLOCKS; }
  if (per_sm < 1) per_sm = 1;
  const unsigned slots = (unsigned)(ctx->sm_count * per_sm);
  // CTAs per wavefront: one when the goals fill the machine; with fewer goals than CTA slots a cluster of CTAs shares a
  // wavefront so that the SMs do not idle (strong scaling across GPUs hands every rank a fraction of the batch)
  int cs = ctx->batch_cluster;
  if (cs <= 0) { cs = 1; while (cs < 8 && (unsigned)(2 * cs) * n <= slots) cs *= 2; }
  if (cs > 1) per_sm = std::max(1, std::min(per_sm, 2));
  unsigned groups = slots / (unsigned)cs;
  if (groups > n) groups = n;
  if (groups == 0) groups = 1;
  int32_t rc;
  if ((rc = ensure_workspace(ctx, groups)) != MNB_OK) return rc;
  if ((rc = ensure_seeds(ctx, n)) != MNB_OK) return rc;
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  if ((rc = ensure_out(ctx, dev ? 0 : (size_t)n * ctx->V, false)) != MNB_OK) return rc;
  if (ctx->h_cancel) *ctx->h_cancel = 0;
  ctx->infl_labels_valid = false;
  CK(cudaMemcpyAsync(ctx->d_seed_faces, seed_faces, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_seed_pos, seed_pos, 3 * sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->d_next_query, 0, sizeof(unsigned int), ctx->stream));
  CK(cudaMemsetAsync(ctx->ws.ctl, 0, sizeof(GroupCtl) * groups, ctx->stream));
  CvpKernelArgs a{};
  fill_cvp_args(ctx, a);
  a.n_queries = n; a.robot_face = -1; a.cost_limit = cost_limit; a.goal_dist_offset = 0.0;
  a.out_dist = dev ? out_dist : ctx->d_out_dist;
  a.out_pred = nullptr; a.out_dir = nullptr; a.out_cut = nullptr;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  if (legacy) { if ((rc = launch_cvp(ctx, a, cs, groups)) != MNB_OK) return rc; }
  else {
    cudaError_t e;
    const unsigned blocks = groups * (unsigned)cs;
    switch (cs) {
      case 1: e = launch_cluster(k_cvp_batch<1>, a, 1, blocks, MNB_BATCH_THREADS, ctx->stream); break;
      case 2: e = launch_cluster(k_cvp_batch<2>, a, 2, blocks, MNB_BATCH_THREADS, ctx->stream); break;
      case 4: e = launch_cluster(k_cvp_batch<4>, a, 4, blocks, MNB_BATCH_THREADS, ctx->stream); break;
      default: e = launch_cluster(k_cvp_batch<8>, a, 8, blocks, MNB_BATCH_THREADS, ctx->stream); break;
    }
    if (e != cudaSuccess) { ctx->err = std::string("cvp batch launch: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)n * ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
  if ((rc = finish_stats(ctx, groups, 1)) != MNB_OK) return rc;
  if (ctx->h_cancel && *ctx->h_cancel) return MNB_CANCELED;
  return MNB_SUCCESS;
}

static int32_t impl_dijkstra(mnb_ctx* ctx, uint32_t seed_vertex, int64_t robot_vertex, double cost_limit, double goal_dist_offset,
                     float* out_dist, uint32_t* out_pred) {
  if (!ctx || !ctx->V) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "costs not set"; return MNB_E_STATE; }
  if (seed_vertex >= ctx->V) return MNB_INVALID_START;
  if (robot_vertex >= (int64_t)ctx->V) return MNB_INVALID_GOAL;
  CK(cudaSetDevice(ctx->device));
  int32_t rc;
  if ((rc = ensure_workspace(ctx, 1)) != MNB_OK) return rc;
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  if ((rc = ensure_out(ctx, (size_t)ctx->V, true)) != MNB_OK) return rc;
  if (ctx->h_cancel) *ctx->h_cancel = 0;     // dijkstra:238
  ctx->infl_labels_valid = false;
  if ((rc = ensure_adj_tables(ctx)) != MNB_OK) return rc;
  CK(cudaMemsetAsync(ctx->ws.ctl, 0, sizeof(GroupCtl), ctx->stream));
  DijkstraKernelArgs a{};
  a.V = ctx->V; a.adj_ptr = ctx->d_adj_ptr; a.adj_nw = ctx->d_adj_nw; a.cost = ctx->d_cost;
  a.invalid = ctx->has_invalid ? ctx->d_invalid : nullptr; a.ws = ctx->ws; a.seed_vertex = seed_vertex;
  a.robot_vertex = robot_vertex; a.cost_limit = cost_limit; a.goal_dist_offset = goal_dist_offset; a.delta = ctx->delta;
  a.out_dist = (dev && out_dist) ? out_dist : ctx->d_out_dist;
  a.out_pred = (dev && out_pred) ? out_pred : ctx->d_out_pred;
  a.cancel_flag = ctx->d_cancel; a.max_rounds = watchdog_rounds(ctx->V);
  if (robot_vertex >= 0 && (uint32_t)robot_vertex == seed_vertex) {   // dijkstra:252-255: "start == goal" returns before the wave
    // the reference has cleared its maps by then (:241-249): distances +inf (seed 0), every vertex its own predecessor
    MNB_LAUNCH(k_dijkstra_trivial, (ctx->V + 255) / 256, 256, 0, ctx->stream, ctx->V, seed_vertex, a.out_dist, a.out_pred);
    CK(cudaGetLastError());
    if (!dev) {
      if (out_dist) CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
      if (out_pred) CK(cudaMemcpyAsync(out_pred, a.out_pred, sizeof(uint32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stats = mnb_stats{}; ctx->stats.kernel_launches = 1;
    return MNB_SUCCESS;
  }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  cudaError_t e;
  const int cs = ctx->cluster;
  if (cs == -1) {   // single plan on the whole GPU (cooperative launch, one CTA per SM)
    a.delta = ctx->dijkstra_grid_delta; a.ell_adj = ctx->d_ell_adj; a.sweeps = ctx->sweeps; a.hop = ctx->w_mean > 0 ? 1.35f * ctx->w_mean : 0.16f;
    e = launch_cooperative(k_dijkstra_grid, a, (unsigned)ctx->sm_count, 512, ctx->stream);
  } else
  switch (cs) {
    case 1: e = launch_cluster(k_dijkstra<1>, a, 1, 1, ctx->threads, ctx->stream); break;
    case 2: e = launch_cluster(k_dijkstra<2>, a, 2, 2, ctx->threads, ctx->stream); break;
    case 4: e = launch_cluster(k_dijkstra<4>, a, 4, 4, ctx->threads, ctx->stream); break;
    case 8: e = launch_cluster(k_dijkstra<8>, a, 8, 8, ctx->threads, ctx->stream); break;
    default: e = launch_cluster(k_dijkstra<16>, a, 16, 16, ctx->threads, ctx->stream); break;
  }
  if (e != cudaSuccess) { ctx->err = std::string("dijkstra launch: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    if (out_dist) CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_pred) CK(cudaMemcpyAsync(out_pred, a.out_pred, sizeof(uint32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
  }
  uint32_t rp = 0;
  if (robot_vertex >= 0) CK(cudaMemcpyAsync(&rp, a.out_pred + robot_vertex, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if ((rc = finish_stats(ctx, 1, 1)) != MNB_OK) return rc;
  if (ctx->h_cancel && *ctx->h_cancel) return MNB_CANCELED;
  if (robot_vertex >= 0 && rp == (uint32_t)robot_vertex) return MNB_NO_PATH_FOUND;          // dijkstra:358-362
  return MNB_SUCCESS;
}

static int32_t impl_dijkstra_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_vertices, double cost_limit, float* out_dist,
                                   uint32_t* out_pred) {
  if (!ctx || !seed_vertices || !out_dist || !ctx->V || n == 0) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "costs not set"; return MNB_E_STATE; }
  for (uint32_t i = 0; i < n; ++i) if (seed_vertices[i] >= ctx->V) return MNB_INVALID_START;
  CK(cudaSetDevice(ctx->device));
  int per_sm = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_dijkstra_batch<1>, DJB_THREADS, 0));
  per_sm = std::max(1, std::min(per_sm, (int)DJB_MINBLOCKS));
  const unsigned slots = (unsigned)(ctx->sm_count * per_sm);
  // CTAs per goal as in impl_cvp_batch: one when the goals fill the machine, a cluster when there are fewer goals than slots
  int cs = ctx->batch_cluster;
  if (cs <= 0) { cs = 1; while (cs < 8 && (unsigned)(2 * cs) * n <= slots) cs *= 2; }
  unsigned groups = std::max(1u, std::min(slots / (unsigned)cs, n));
  const size_t V = ctx->V;
  if (groups > ctx->djb_groups) {
    dfree(ctx->d_djb_scratch); dfree(ctx->d_djb_ctl); ctx->djb_groups = 0;
    CK(dalloc(&ctx->d_djb_scratch, (size_t)groups * 3 * V)); CK(dalloc(&ctx->d_djb_ctl, (size_t)groups));
    ctx->djb_groups = groups;
  }
  if (n > ctx->djb_seed_cap) { dfree(ctx->d_djb_seeds); ctx->djb_seed_cap = 0; CK(dalloc(&ctx->d_djb_seeds, (size_t)n)); ctx->djb_seed_cap = n; }
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  int32_t rc;
  if (!dev) {
    if ((rc = ensure_out(ctx, (size_t)n * V, false)) != MNB_OK) return rc;
    if (out_pred && (size_t)n * V > ctx->djb_pred_cap) {
      dfree(ctx->d_djb_pred); ctx->djb_pred_cap = 0; CK(dalloc(&ctx->d_djb_pred, (size_t)n * V)); ctx->djb_pred_cap = (size_t)n * V;
    }
  }
  if ((rc = ensure_adj_tables(ctx)) != MNB_OK) return rc;
  if (ctx->h_cancel) *ctx->h_cancel = 0;
  CK(cudaMemcpyAsync(ctx->d_djb_seeds, seed_vertices, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->d_next_query, 0, sizeof(unsigned int), ctx->stream));
  CK(cudaMemsetAsync(ctx->d_djb_ctl, 0, sizeof(GroupCtl) * groups, ctx->stream));
  DijkstraBatchArgs a{};
  a.V = ctx->V; a.adj_ptr = ctx->d_adj_ptr; a.adj_nw = ctx->d_adj_nw; a.ell_adj = ctx->d_ell_adj;
  a.cost = ctx->d_cost; a.invalid = ctx->has_invalid ? ctx->d_invalid : nullptr; a.cost_limit = cost_limit;
  a.delta = ctx->delta; a.n_queries = n; a.seeds = ctx->d_djb_seeds;
  a.out_dist = dev ? out_dist : ctx->d_out_dist;
  a.out_pred = !out_pred ? nullptr : (dev ? out_pred : ctx->d_djb_pred);
  a.scratch = ctx->d_djb_scratch; a.ctl = ctx->d_djb_ctl; a.next_query = ctx->d_next_query; a.cancel_flag = ctx->d_cancel;
  a.max_rounds = watchdog_rounds(ctx->V);
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  cudaError_t e;
  const unsigned blocks = groups * (unsigned)cs;
  switch (cs) {
    case 1: e = launch_cluster(k_dijkstra_batch<1>, a, 1, blocks, DJB_THREADS, ctx->stream); break;
    case 2: e = launch_cluster(k_dijkstra_batch<2>, a, 2, blocks, DJB_THREADS, ctx->stream); break;
    case 4: e = launch_cluster(k_dijkstra_batch<4>, a, 4, blocks, DJB_THREADS, ctx->stream); break;
    default: e = launch_cluster(k_dijkstra_batch<8>, a, 8, blocks, DJB_THREADS, ctx->stream); break;
  }
  if (e != cudaSuccess) { ctx->err = std::string("dijkstra batch launch: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)n * V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_pred) CK(cudaMemcpyAsync(out_pred, a.out_pred, sizeof(uint32_t) * (size_t)n * V, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if ((rc = finish_stats(ctx, groups, 1, ctx->d_djb_ctl)) != MNB_OK) return rc;
  if (ctx->h_cancel && *ctx->h_cancel) return MNB_CANCELED;
  return MNB_SUCCESS;
}

int32_t mnb_get_vertex_normals(mnb_ctx* ctx, float* out) {
  if (!ctx || !out || !ctx->V) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(out, ctx->d_vertex_normals, sizeof(float) * 3 * (size_t)ctx->V, out_kind(ctx), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

static int32_t impl_compute_layers(mnb_ctx* ctx, const mnb_layer_params* params, const float* clearance, float* out_costs,
                           float* out_combined, uint8_t* out_lethal_mask) {
  if (!ctx || !params || !ctx->V) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  const size_t V = ctx->V;
  if (!ctx->d_layer_costs) {
    CK(dalloc(&ctx->d_layer_costs, 6 * V)); CK(dalloc(&ctx->d_layer_combined, V)); CK(dalloc(&ctx->d_layer_mask, V));
    CK(dalloc(&ctx->d_overflow, (size_t)1));
  }
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  if (clearance) {
    if (!ctx->d_clearance) CK(dalloc(&ctx->d_clearance, V));
    CK(cudaMemcpyAsync(ctx->d_clearance, clearance, sizeof(float) * V, in_kind(ctx), ctx->stream));
  }
  CK(cudaMemsetAsync(ctx->d_overflow, 0, sizeof(unsigned int), ctx->stream));
  LayerKernelArgs a{};
  a.V = ctx->V; a.pos = ctx->d_pos; a.vn = ctx->d_vertex_normals; a.adj_ptr = ctx->d_adj_ptr; a.adj_nbr = ctx->d_adj_nbr;
  a.border = ctx->d_border; a.clearance = clearance ? ctx->d_clearance : nullptr; a.P = *params;
  a.costs = (dev && out_costs) ? out_costs : ctx->d_layer_costs;
  a.combined = (dev && out_combined) ? out_combined : ctx->d_layer_combined;
  a.lethal_mask = (dev && out_lethal_mask) ? out_lethal_mask : ctx->d_layer_mask;
  a.overflow = ctx->d_overflow;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  if (ctx->layers_smem) {
    if (!ctx->d_pos4) {
      CK(dalloc(&ctx->d_pos4, V)); CK(dalloc(&ctx->d_vn4, V)); CK(dalloc(&ctx->d_nbr8, 8 * V));
      MNB_LAUNCH(k_pack_layers, (ctx->V + 255) / 256, 256, 0, ctx->stream, (const float*)ctx->d_pos, (const float*)ctx->d_vertex_normals,
                 (const uint32_t*)ctx->d_adj_ptr, (const uint32_t*)ctx->d_adj_nbr, ctx->V, ctx->d_pos4, ctx->d_vn4, ctx->d_nbr8);
      CK(cudaGetLastError());
    }
    a.pos4 = ctx->d_pos4; a.vn4 = ctx->d_vn4; a.nbr8 = reinterpret_cast<const uint4*>(ctx->d_nbr8);
    if (ctx->layers_smem == 8 || ctx->layers_smem == 9) {      // walk_pf16 compiled for more resident CTAs (fewer registers): 8 -> 64 x 12, 9 -> 128 x 6
      const int T = ctx->layers_smem == 8 ? 64 : 128;
      const size_t smem = (size_t)(2 * NB_HASH + LS_STACK) * T;
      if (T == 64) { CK(cudaFuncSetAttribute(k_layers_pf16<64, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH((k_layers_pf16<64, 12>), (ctx->V + 63) / 64, 64, smem, ctx->stream, a); }
      else { CK(cudaFuncSetAttribute(k_layers_pf16<128, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH((k_layers_pf16<128, 6>), (ctx->V + 127) / 128, 128, smem, ctx->stream, a); }
    } else
    if (ctx->layers_smem >= 5) {            // walk_pf16 (16-bit seen-set): 5 -> 64 threads per CTA, 6 -> 128, 7 -> 256
      const int T = ctx->layers_smem == 5 ? 64 : (ctx->layers_smem == 6 ? 128 : 256);
      const size_t smem = (size_t)(2 * NB_HASH + LS_STACK) * T;
      if (T == 64) { CK(cudaFuncSetAttribute(k_layers_pf16<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf16<64>, (ctx->V + 63) / 64, 64, smem, ctx->stream, a); }
      else if (T == 128) { CK(cudaFuncSetAttribute(k_layers_pf16<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf16<128>, (ctx->V + 127) / 128, 128, smem, ctx->stream, a); }
      else { CK(cudaFuncSetAttribute(k_layers_pf16<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf16<256>, (ctx->V + 255) / 256, 256, smem, ctx->stream, a); }
    } else
    if (ctx->layers_smem >= 2) {            // walk_pf: 2 -> 64 threads per CTA, 3 -> 128, 4 -> 32
      const int T = ctx->layers_smem == 2 ? 64 : (ctx->layers_smem == 3 ? 128 : 32);
      const size_t smem = sizeof(uint32_t) * (size_t)(NB_HASH + LS_STACK) * T;
      if (T == 64) { CK(cudaFuncSetAttribute(k_layers_pf<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf<64>, (ctx->V + 63) / 64, 64, smem, ctx->stream, a); }
      else if (T == 128) { CK(cudaFuncSetAttribute(k_layers_pf<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf<128>, (ctx->V + 127) / 128, 128, smem, ctx->stream, a); }
      else { CK(cudaFuncSetAttribute(k_layers_pf<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); MNB_LAUNCH(k_layers_pf<32>, (ctx->V + 31) / 32, 32, smem, ctx->stream, a); }
    } else {
    const size_t smem = sizeof(uint32_t) * (size_t)(NB_HASH + LS_STACK) * LS_THREADS;       // 88 KB: two CTAs per SM
    CK(cudaFuncSetAttribute(k_layers<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MNB_LAUNCH(k_layers<true>, (ctx->V + LS_THREADS - 1) / LS_THREADS, LS_THREADS, smem, ctx->stream, a);
    }
  } else {
    MNB_LAUNCH(k_layers<false>, (ctx->V + 127) / 128, 128, 0, ctx->stream, a);
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    if (out_costs) CK(cudaMemcpyAsync(out_costs, a.costs, sizeof(float) * 6 * V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_combined) CK(cudaMemcpyAsync(out_combined, a.combined, sizeof(float) * V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_lethal_mask) CK(cudaMemcpyAsync(out_lethal_mask, a.lethal_mask, V, cudaMemcpyDeviceToHost, ctx->stream));
  }
  unsigned int ovf = 0;
  CK(cudaMemcpyAsync(&ovf, ctx->d_overflow, sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = 1; ctx->stats.settled = ctx->V;
  if (ovf) { ctx->err = "layer neighbourhood exceeds the per-vertex scratch (radius too large for the mesh resolution)"; return MNB_E_NOMEM; }
  return MNB_OK;
}

static int32_t impl_vector_map(mnb_ctx* ctx, const uint32_t* pred, const float* direction, const int32_t* cutting_face, float* out_vec) {
  if (!ctx || !ctx->V || !out_vec) return MNB_E_ARG;
  if (!pred && !ctx->last_valid) { ctx->err = "mnb_vector_map(pred = NULL) needs a successful mnb_cvp on this context first"; return MNB_E_STATE; }
  CK(cudaSetDevice(ctx->device));
  const size_t V = ctx->V;
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  const uint32_t* d_pred = pred; const float* d_dir = direction; const int32_t* d_cut = cutting_face; float* d_out = out_vec;
  float* tmp_out = nullptr; uint32_t* tmp_pred = nullptr; float* tmp_dir = nullptr; int32_t* tmp_cut = nullptr;
  if (!pred) {            // the device-resident result of the last CVP plan (nothing is uploaded)
    d_pred = ctx->last_pred; d_dir = ctx->last_dir; d_cut = ctx->last_cut;
    if (!dev) { CK(dalloc(&tmp_out, 3 * V)); d_out = tmp_out; }
  } else if (!dev) {
    CK(dalloc(&tmp_out, 3 * V)); CK(dalloc(&tmp_pred, V));
    CK(cudaMemcpyAsync(tmp_pred, pred, sizeof(uint32_t) * V, cudaMemcpyHostToDevice, ctx->stream));
    d_pred = tmp_pred; d_out = tmp_out;
    if (direction) { CK(dalloc(&tmp_dir, V)); CK(cudaMemcpyAsync(tmp_dir, direction, sizeof(float) * V, cudaMemcpyHostToDevice, ctx->stream)); d_dir = tmp_dir; }
    if (cutting_face) { CK(dalloc(&tmp_cut, V)); CK(cudaMemcpyAsync(tmp_cut, cutting_face, sizeof(int32_t) * V, cudaMemcpyHostToDevice, ctx->stream)); d_cut = tmp_cut; }
  }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  MNB_LAUNCH(k_vector_map, (ctx->V + 255) / 256, 256, 0, ctx->stream, ctx->d_pos, ctx->d_vertex_normals, d_pred, d_dir, d_cut, ctx->V, d_out);
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) CK(cudaMemcpyAsync(out_vec, d_out, sizeof(float) * 3 * V, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  dfree(tmp_out); dfree(tmp_pred); dfree(tmp_dir); dfree(tmp_cut);
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = 1; ctx->stats.settled = ctx->V;
  return MNB_OK;
}

static int32_t impl_cvp_backtrack(mnb_ctx* ctx, const float robot_pos[3], uint32_t robot_face, double step_width, uint32_t max_points,
                          float* path_pos, uint32_t* path_face, uint32_t* n_points) {
  if (!ctx || !ctx->V || !robot_pos || !path_pos || !n_points || max_points < 2) return MNB_E_ARG;
  if (!ctx->last_valid) { ctx->err = "mnb_cvp_backtrack needs a preceding successful mnb_cvp on this context"; return MNB_E_STATE; }
  if (robot_face >= ctx->F) return MNB_INVALID_GOAL;
  CK(cudaSetDevice(ctx->device));
  if (max_points > ctx->path_cap) {
    dfree(ctx->d_path_pos); dfree(ctx->d_path_face); ctx->path_cap = 0;
    CK(dalloc(&ctx->d_path_pos, 3 * (size_t)max_points)); CK(dalloc(&ctx->d_path_face, (size_t)max_points));
    ctx->path_cap = max_points;
  }
  if (!ctx->d_bt_result) CK(dalloc(&ctx->d_bt_result, (size_t)2));
  BacktrackArgs a{};
  a.pos = ctx->d_pos; a.vn = ctx->d_vertex_normals; a.faces = ctx->d_faces; a.cor_ptr = ctx->d_cor_ptr; a.cor_idx = ctx->d_cor_idx;
  a.pred = ctx->last_pred; a.direction = ctx->last_dir; a.cut = ctx->last_cut;
  for (int k = 0; k < 3; ++k) { a.start[k] = ctx->last_seed_pos[k]; a.goal[k] = robot_pos[k]; }
  a.start_face = ctx->last_seed_face; a.goal_face = robot_face; a.step_width = step_width; a.max_points = max_points;
  a.path_pos = ctx->d_path_pos; a.path_face = ctx->d_path_face; a.result = ctx->d_bt_result; a.cancel_flag = ctx->d_cancel;
  a.layer = RepulsiveField{};
  if (ctx->repulsive_on && ctx->infl_field_valid) a.layer = repulsive_field_of(ctx);
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  CK(cudaFuncSetAttribute(k_backtrack, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BtShared)));
  MNB_LAUNCH(k_backtrack, 1, 32, sizeof(BtShared), ctx->stream, a);
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  int32_t res[2] = {0, 0};
  CK(cudaMemcpyAsync(res, ctx->d_bt_result, sizeof(res), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const uint32_t n = (uint32_t)res[1] < max_points ? (uint32_t)res[1] : max_points;
  *n_points = n;
  const cudaMemcpyKind kind = ctx->ptr_mode == MNB_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  CK(cudaMemcpyAsync(path_pos, ctx->d_path_pos, sizeof(float) * 3 * (size_t)n, kind, ctx->stream));
  if (path_face) CK(cudaMemcpyAsync(path_face, ctx->d_path_face, sizeof(uint32_t) * (size_t)n, kind, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = 1; ctx->stats.settled = n;
  if (res[0] == MNB_E_STATE) { ctx->err = "back-tracking exceeded max_points (cyclic vector field?) or the face search list"; return MNB_E_STATE; }
  return res[0];
}

static int32_t impl_locate(mnb_ctx* ctx, uint32_t n, const float* points, uint32_t* out_vertex, int32_t* out_face, float* out_bary) {
  if (!ctx || !ctx->V || !points || n == 0) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  float* d_pts = nullptr; unsigned long long* d_keys = nullptr; uint32_t* d_v = nullptr; int32_t* d_f = nullptr; float* d_b = nullptr;
  CK(dalloc(&d_keys, (size_t)n));
  CK(cudaMemsetAsync(d_keys, 0xff, sizeof(unsigned long long) * (size_t)n, ctx->stream));
  const float* pts = points;
  if (!dev) {
    CK(dalloc(&d_pts, 3 * (size_t)n)); CK(dalloc(&d_v, (size_t)n)); CK(dalloc(&d_f, (size_t)n)); CK(dalloc(&d_b, 3 * (size_t)n));
    CK(cudaMemcpyAsync(d_pts, points, sizeof(float) * 3 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    pts = d_pts;
  }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  const uint32_t want = (ctx->V + 255) / 256, cap = (uint32_t)ctx->sm_count * 8;
  const uint32_t blocks = want < cap ? want : cap;
  uint32_t launches = 0;
  for (uint32_t q0 = 0; q0 < n; q0 += LOC_Q, ++launches)
    MNB_LAUNCH(k_nearest_vertex, blocks, 256, 0, ctx->stream, ctx->d_pos, ctx->V, pts, q0, n - q0 < (uint32_t)LOC_Q ? n - q0 : (uint32_t)LOC_Q, d_keys);
  MNB_LAUNCH(k_containing_face, (n + 127) / 128, 128, 0, ctx->stream, ctx->d_pos, ctx->d_faces, ctx->d_cor_ptr, ctx->d_cor_idx, pts, n, d_keys,
                                                           dev ? out_vertex : d_v, dev ? out_face : d_f, dev ? out_bary : d_b);
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    if (out_vertex) CK(cudaMemcpyAsync(out_vertex, d_v, sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_face) CK(cudaMemcpyAsync(out_face, d_f, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_bary) CK(cudaMemcpyAsync(out_bary, d_b, sizeof(float) * 3 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  dfree(d_pts); dfree(d_keys); dfree(d_v); dfree(d_f); dfree(d_b);
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = launches + 1; ctx->stats.settled = n;
  return MNB_OK;
}

// experiment knob (not part of the public header): in-round sweeps of the whole-grid single-plan kernel
int32_t mnb_debug_set_sweeps(mnb_ctx* ctx, int32_t k) { if (!ctx || k < -1 || k > 64) return MNB_E_ARG; ctx->sweeps = k; return MNB_OK; }

int32_t mnb_debug_set_grid_engine(mnb_ctx* ctx, int32_t mode, float delta_w) { if (!ctx) return MNB_E_ARG; ctx->grid_engine = mode; if (delta_w > 0) ctx->grid2_delta_w = delta_w; return MNB_OK; }
int32_t mnb_debug_set_infl_skip(mnb_ctx* ctx, int32_t on) { if (!ctx) return MNB_E_ARG; ctx->infl_skip_clean = on != 0; return MNB_OK; }
int32_t mnb_debug_set_layers_smem(mnb_ctx* ctx, int32_t mode) { if (!ctx || mode < 0 || mode > 9) return MNB_E_ARG; ctx->layers_smem = mode; ctx->layers_explicit = true; return MNB_OK; }
int32_t mnb_debug_set_skip_clean(mnb_ctx* ctx, int32_t on) { if (!ctx) return MNB_E_ARG; ctx->skip_clean = on != 0; ctx->grid_blocks_per_sm = 0; return MNB_OK; }

// debugging aid (not part of the public header): raw labels {d, a1, a2, a3|flag} of wavefront group 0
int32_t mnb_debug_get_labels(mnb_ctx* ctx, uint32_t* out4v) {
  if (!ctx || !ctx->ws.state) return MNB_E_ARG;
  CK(cudaMemcpy(out4v, ctx->ws.state, sizeof(uint4) * (size_t)ctx->V, cudaMemcpyDeviceToHost));
  return MNB_OK;
}

// debugging aid (not part of the public header): side arrays of the labels of wavefront group 0 (level-1 ids, ext words,
// the first n_pool words of the level pool) -- tools/emu_pop_order.py rebuilds every vertex' level stack from them
int32_t mnb_debug_get_label_sides(mnb_ctx* ctx, uint32_t* root, uint32_t* ext, uint32_t* pool, uint32_t n_pool) {
  if (!ctx || !ctx->ws.state) return MNB_E_ARG;
  CK(cudaMemcpy(root, ctx->ws.root, sizeof(uint32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(ext, ctx->ws.ext, sizeof(uint32_t) * (size_t)ctx->V, cudaMemcpyDeviceToHost));
  if (n_pool) CK(cudaMemcpy(pool, ctx->ws.pool, sizeof(uint32_t) * (size_t)std::min<uint32_t>(n_pool, ctx->ws.pool_cap), cudaMemcpyDeviceToHost));
  return MNB_OK;
}

}  // extern "C"

// InflationLayer::waveCostInflation; with want_update additionally the update set of InflationLayer::onInputChanged
static int32_t inflate_impl(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid,
                            const mnb_inflation_params* params, float* out_dist, float* out_cost, bool want_update,
                            uint32_t* out_changed, uint32_t* n_changed) {
  if (!ctx || !ctx->V || !params || (n && !lethals)) return MNB_E_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->infl_labels_valid = false;
  int32_t rc;
  if ((rc = ensure_workspace(ctx, 1)) != MNB_OK) return rc;
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  if ((rc = ensure_out(ctx, (size_t)ctx->V, false)) != MNB_OK) return rc;
  if (!ctx->d_out_cost) CK(dalloc(&ctx->d_out_cost, (size_t)ctx->V));
  if (n > ctx->lethal_cap) { dfree(ctx->d_lethals); CK(dalloc(&ctx->d_lethals, (size_t)n)); ctx->lethal_cap = n; }
  if (n) CK(cudaMemcpyAsync(ctx->d_lethals, lethals, sizeof(uint32_t) * n, in_kind(ctx), ctx->stream));
  if (invalid) {
    if (!ctx->d_infl_invalid) CK(dalloc(&ctx->d_infl_invalid, (size_t)ctx->V));
    CK(cudaMemcpyAsync(ctx->d_infl_invalid, invalid, (size_t)ctx->V, in_kind(ctx), ctx->stream));
  }
  CK(cudaMemsetAsync(ctx->ws.ctl, 0, sizeof(GroupCtl), ctx->stream));
  InflateKernelArgs a{};
  a.V = ctx->V; a.cor_ptr = ctx->d_cor_ptr; a.cor_idx = ctx->d_cor_idx; a.cor_wd = ctx->d_cor_wd; a.cor_eid = ctx->d_cor_eid;
  a.invalid = invalid ? ctx->d_infl_invalid : nullptr; a.ws = ctx->ws; a.lethals = ctx->d_lethals; a.n_lethals = n;
  a.max_distance = (float)params->inflation_radius;      // double -> `const float&` parameter (inflation_layer.cpp:240,450)
  a.params.inscribed_radius = params->inscribed_radius; a.params.inflation_radius = params->inflation_radius;
  a.params.lethal_value = params->lethal_value; a.params.inscribed_value = params->inscribed_value;
  a.params.cost_scaling_factor = params->cost_scaling_factor;
  a.out_dist = (dev && out_dist) ? out_dist : ctx->d_out_dist;
  a.out_cost = (dev && out_cost) ? out_cost : ctx->d_out_cost;
  a.max_rounds = watchdog_rounds(ctx->V); a.skip_clean = ctx->infl_skip_clean;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  int infl_per_sm = 1;
  if (MNB_INFL_MINBLOCKS > 1) {
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&infl_per_sm, k_inflate, ctx->threads, 0));
    infl_per_sm = std::max(1, std::min(infl_per_sm, (int)MNB_INFL_MINBLOCKS));
  }
  CK(launch_cooperative(k_inflate, a, (unsigned)(ctx->sm_count * infl_per_sm), ctx->threads, ctx->stream));
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  if (!dev) {
    if (out_dist) CK(cudaMemcpyAsync(out_dist, a.out_dist, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
    if (out_cost) CK(cudaMemcpyAsync(out_cost, a.out_cost, sizeof(float) * (size_t)ctx->V, cudaMemcpyDeviceToHost, ctx->stream));
  }
  int32_t rc2 = finish_stats(ctx, 1, 1);
  if (rc2 != MNB_OK) return rc2;
  // the riskiness map of this run is the "previous" one of the next mnb_inflation_update (riskiness_ = std::move(new_costs))
  const size_t V = ctx->V;
  if (want_update) {
    const uint32_t n_tiles = (uint32_t)((V + US_TILE - 1) / US_TILE);
    if (!ctx->d_changed) { CK(dalloc(&ctx->d_changed, V)); CK(dalloc(&ctx->d_tile_count, (size_t)n_tiles)); CK(dalloc(&ctx->d_total, (size_t)1)); }
    const float* old = ctx->prev_risk_valid ? ctx->d_prev_risk : nullptr;
    uint32_t* d_out = (dev && out_changed) ? out_changed : ctx->d_changed;
    MNB_LAUNCH(k_update_set_count, n_tiles, 256, 0, ctx->stream, (const float*)a.out_cost, old, ctx->V, ctx->d_tile_count);
    MNB_LAUNCH(k_update_set_scan, 1, 1024, 0, ctx->stream, ctx->d_tile_count, n_tiles, ctx->d_total);
    MNB_LAUNCH(k_update_set_write, n_tiles, 256, 0, ctx->stream, (const float*)a.out_cost, old, ctx->V, (const unsigned int*)ctx->d_tile_count, d_out);
    CK(cudaGetLastError());
    unsigned int total = 0;
    CK(cudaMemcpyAsync(&total, ctx->d_total, sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (n_changed) *n_changed = total;
    if (!dev && out_changed && total) CK(cudaMemcpyAsync(out_changed, d_out, sizeof(uint32_t) * (size_t)total, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.kernel_launches += 3;
  }
  if (!ctx->d_prev_risk) CK(dalloc(&ctx->d_prev_risk, V));
  CK(cudaMemcpyAsync(ctx->d_prev_risk, a.out_cost, sizeof(float) * V, cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->prev_risk_valid = true;
  ctx->infl_labels_valid = true; ctx->infl_had_invalid = invalid != nullptr; ctx->infl_params = *params; ctx->infl_field_valid = false; ctx->infl_rounds = ctx->stats.rounds;
  if (!ctx->d_infl_dist) CK(dalloc(&ctx->d_infl_dist, V));
  CK(cudaMemcpyAsync(ctx->d_infl_dist, a.out_dist, sizeof(float) * V, cudaMemcpyDeviceToDevice, ctx->stream));   // distances_
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

extern "C" {

static int32_t impl_inflate(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid,
                    const mnb_inflation_params* params, float* out_dist, float* out_cost) {
  return inflate_impl(ctx, lethals, n, invalid, params, out_dist, out_cost, false, nullptr, nullptr);
}

static int32_t impl_inflation_update(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid,
                             const mnb_inflation_params* params, float* out_dist, float* out_cost, uint32_t* out_changed,
                             uint32_t* n_changed) {
  if (!n_changed) return MNB_E_ARG;
  return inflate_impl(ctx, lethals, n, invalid, params, out_dist, out_cost, true, out_changed, n_changed);
}

int32_t mnb_get_costs(mnb_ctx* ctx, float* out_vertex_costs, float* out_edge_weights) {
  if (!ctx || !ctx->V) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "costs not set"; return MNB_E_STATE; }
  CK(cudaSetDevice(ctx->device));
  if (out_vertex_costs) CK(cudaMemcpyAsync(out_vertex_costs, ctx->d_cost, sizeof(float) * (size_t)ctx->V, out_kind(ctx), ctx->stream));
  if (out_edge_weights) CK(cudaMemcpyAsync(out_edge_weights, ctx->d_edge_w, sizeof(float) * (size_t)ctx->E, out_kind(ctx), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return MNB_OK;
}

static int32_t impl_update_vertex_costs(mnb_ctx* ctx, uint32_t n_changed, const uint32_t* changed, const float* costs,
                                int32_t costs_indexed_by_vertex, float default_value, double edge_cost_factor) {
  if (!ctx || !ctx->V || (n_changed && (!changed || !costs))) return MNB_E_ARG;
  if (!ctx->costs_set) { ctx->err = "mnb_update_vertex_costs needs mnb_set_costs / mnb_compute_edge_weights first"; return MNB_E_STATE; }
  if (n_changed == 0) return MNB_OK;
  CK(cudaSetDevice(ctx->device));
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  const uint32_t* d_ids = changed; const float* d_costs = costs;
  if (!dev) {
    const size_t nc = costs_indexed_by_vertex ? (size_t)ctx->V : (size_t)n_changed;
    if (n_changed > ctx->upd_cap) { dfree(ctx->d_upd_ids); ctx->upd_cap = 0; CK(dalloc(&ctx->d_upd_ids, (size_t)n_changed)); ctx->upd_cap = n_changed; }
    if (nc > ctx->upd_cost_cap) { dfree(ctx->d_upd_costs); ctx->upd_cost_cap = 0; CK(dalloc(&ctx->d_upd_costs, nc)); ctx->upd_cost_cap = nc; }
    CK(cudaMemcpyAsync(ctx->d_upd_ids, changed, sizeof(uint32_t) * (size_t)n_changed, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_upd_costs, costs, sizeof(float) * nc, cudaMemcpyHostToDevice, ctx->stream));
    d_ids = ctx->d_upd_ids; d_costs = ctx->d_upd_costs;
  }
  if (!ctx->d_upd_stamp || ctx->upd_call == 0xffffffffu) {
    if (!ctx->d_upd_stamp) CK(dalloc(&ctx->d_upd_stamp, (size_t)ctx->V));
    CK(cudaMemsetAsync(ctx->d_upd_stamp, 0, sizeof(uint32_t) * (size_t)ctx->V, ctx->stream));
    ctx->upd_call = 0;
  }
  ++ctx->upd_call;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  unsigned launches = 1;
  MNB_LAUNCH(k_update_costs, (n_changed + 255) / 256, 256, 0, ctx->stream, d_ids, n_changed, d_costs, (int)(costs_indexed_by_vertex != 0),
             default_value, ctx->V, ctx->d_cost, ctx->d_upd_stamp, ctx->upd_call);
  if (edge_cost_factor != 0) {                       // mesh_map.cpp:568-572: no edge update at all for a zero factor
    const unsigned blocks = (unsigned)(((size_t)n_changed * ELL_W + 255) / 256);
    MNB_LAUNCH(k_update_edge_weights, blocks, 256, 0, ctx->stream, d_ids, n_changed, ctx->V, (const uint32_t*)ctx->d_adj_ptr,
               (const uint32_t*)ctx->d_adj_eid, (const uint32_t*)ctx->d_edges, (const float*)ctx->d_cost, (const float*)ctx->d_edge_dist,
               edge_cost_factor, ctx->d_edge_w);
    RefreshArgs r{};
    r.changed = d_ids; r.n = n_changed; r.V = ctx->V; r.faces = ctx->d_faces; r.cor_ptr = ctx->d_cor_ptr; r.cor_idx = ctx->d_cor_idx;
    r.cor_eid = ctx->d_cor_eid; r.face_cor = ctx->d_face_cor; r.adj_ptr = ctx->d_adj_ptr; r.adj_nbr = ctx->d_adj_nbr; r.adj_eid = ctx->d_adj_eid; r.w = ctx->d_edge_w;
    r.cor_w = ctx->d_cor_w; r.ell_w = ctx->d_ell_w; r.ell_geo = ctx->d_ell_geo;
    r.adj_nw = ctx->adj_dirty ? nullptr : ctx->d_adj_nw; r.ell_adj = ctx->adj_dirty ? nullptr : ctx->d_ell_adj;   // stale tables are rebuilt whole anyway
    r.stamp = ctx->d_upd_stamp; r.call = ctx->upd_call;
    MNB_LAUNCH(k_refresh_weight_tables, blocks, 256, 0, ctx->stream, r);
    launches = 3;
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = launches; ctx->stats.settled = n_changed;
  return MNB_OK;
}

}  // extern "C"

static int32_t combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                  const float* weights /* null: MaxCombinationLayer */, const uint8_t* const* layer_lethal,
                                  uint32_t n_changed, const uint32_t* changed, float* io_costs, uint8_t* io_lethal) {
  if (!ctx || !ctx->V || n_layers == 0 || n_layers > (uint32_t)COMB_MAX_LAYERS || !layer_costs || !defaults || !io_costs ||
      (n_changed && !changed)) return MNB_E_ARG;
  for (uint32_t l = 0; l < n_layers; ++l) if (!layer_costs[l]) return MNB_E_ARG;
  if (n_changed == 0) return MNB_OK;
  CK(cudaSetDevice(ctx->device));
  const bool dev = ctx->ptr_mode == MNB_PTR_DEVICE;
  const size_t V = ctx->V;
  CombineArgs a{};
  a.n_layers = n_layers; a.n = n_changed; a.V = ctx->V; a.average = weights ? 1 : 0;
  for (uint32_t l = 0; l < n_layers; ++l) a.weight[l] = weights ? weights[l] : 1.0f;
  std::vector<void*> tmp;                             // host-pointer mode: device copies of the maps
  auto cleanup = [&]() { for (void* q : tmp) cudaFree(q); };
  auto up = [&](const void* h, size_t bytes, void** d) -> cudaError_t {
    cudaError_t e = cudaMalloc(d, bytes ? bytes : 1); if (e != cudaSuccess) return e;
    tmp.push_back(*d);
    return cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, ctx->stream);
  };
  cudaError_t e = cudaSuccess;
  for (uint32_t l = 0; l < n_layers && e == cudaSuccess; ++l) {
    a.def[l] = defaults[l];
    if (dev) { a.costs[l] = layer_costs[l]; a.lethal[l] = layer_lethal ? layer_lethal[l] : nullptr; continue; }
    void* d = nullptr;
    e = up(layer_costs[l], sizeof(float) * V, &d); a.costs[l] = (const float*)d;
    if (e == cudaSuccess && layer_lethal && layer_lethal[l]) { e = up(layer_lethal[l], V, &d); a.lethal[l] = (const uint8_t*)d; }
  }
  void* d_ids = nullptr; void* d_io = nullptr; void* d_il = nullptr;
  if (!dev && e == cudaSuccess) {
    e = up(changed, sizeof(uint32_t) * (size_t)n_changed, &d_ids);
    if (e == cudaSuccess) e = up(io_costs, sizeof(float) * V, &d_io);
    if (e == cudaSuccess && io_lethal) e = up(io_lethal, V, &d_il);
  }
  if (e != cudaSuccess) { cleanup(); ctx->err = std::string("mnb_max_combination_update: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  a.changed = dev ? changed : (const uint32_t*)d_ids;
  a.io_costs = dev ? io_costs : (float*)d_io;
  a.io_lethal = dev ? io_lethal : (uint8_t*)d_il;
  cudaEventRecord(ctx->ev0, ctx->stream);
  MNB_LAUNCH(k_max_combination_update, (n_changed + 255) / 256, 256, 0, ctx->stream, a);
  e = cudaGetLastError();
  cudaEventRecord(ctx->ev1, ctx->stream);
  if (e == cudaSuccess && !dev) {
    e = cudaMemcpyAsync(io_costs, a.io_costs, sizeof(float) * V, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && io_lethal) e = cudaMemcpyAsync(io_lethal, a.io_lethal, V, cudaMemcpyDeviceToHost, ctx->stream);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cleanup();
  if (e != cudaSuccess) { ctx->err = std::string("mnb_max_combination_update: ") + cudaGetErrorString(e); return MNB_E_CUDA; }
  float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats = mnb_stats{}; ctx->stats.kernel_ms = ms; ctx->stats.kernel_launches = 1; ctx->stats.settled = n_changed;
  return MNB_OK;
}

extern "C" {

static int32_t impl_max_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const uint8_t* const* layer_lethal, uint32_t n_changed, const uint32_t* changed,
                                   float* io_costs, uint8_t* io_lethal) {
  return combination_update(ctx, n_layers, layer_costs, defaults, nullptr, layer_lethal, n_changed, changed, io_costs, io_lethal);
}

static int32_t impl_avg_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const float* weights, const uint8_t* const* layer_lethal, uint32_t n_changed,
                                   const uint32_t* changed, float* io_costs, uint8_t* io_lethal) {
  if (!weights) return MNB_E_ARG;
  return combination_update(ctx, n_layers, layer_costs, defaults, weights, layer_lethal, n_changed, changed, io_costs, io_lethal);
}

// ---- exception barrier: nothing propagates through the C ABI; a failed call leaves no half-built state behind ----
int32_t mnb_set_mesh(mnb_ctx* ctx, uint32_t V, uint32_t F, const float* pos, const uint32_t* faces,
                     const uint32_t* edges, uint32_t E) {
  const int32_t rc = guarded(ctx, [&]() { return impl_set_mesh(ctx, V, F, pos, faces, edges, E); });
  if (rc != MNB_OK && ctx) { free_mesh(ctx); ctx->V = 0; ctx->F = 0; ctx->E = 0; }      // no half-built context
  return rc;
}
int32_t mnb_cvp(mnb_ctx* ctx, uint32_t seed_face, const float seed_pos[3], int64_t robot_face, double cost_limit,
                double goal_dist_offset, float* out_dist, uint32_t* out_pred, float* out_direction, int32_t* out_cut) {
  return guarded(ctx, [&]() { return impl_cvp(ctx, seed_face, seed_pos, robot_face, cost_limit, goal_dist_offset, out_dist, out_pred, out_direction, out_cut); });
}
int32_t mnb_cvp_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_faces, const float* seed_pos, double cost_limit,
                      float* out_dist) {
  return guarded(ctx, [&]() { return impl_cvp_batch(ctx, n, seed_faces, seed_pos, cost_limit, out_dist); });
}
int32_t mnb_dijkstra(mnb_ctx* ctx, uint32_t seed_vertex, int64_t robot_vertex, double cost_limit, double goal_dist_offset,
                     float* out_dist, uint32_t* out_pred) {
  return guarded(ctx, [&]() { return impl_dijkstra(ctx, seed_vertex, robot_vertex, cost_limit, goal_dist_offset, out_dist, out_pred); });
}
int32_t mnb_dijkstra_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_vertices, double cost_limit, float* out_dist, uint32_t* out_pred) {
  return guarded(ctx, [&]() { return impl_dijkstra_batch(ctx, n, seed_vertices, cost_limit, out_dist, out_pred); });
}
int32_t mnb_inflate(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid,
                    const mnb_inflation_params* params, float* out_dist, float* out_cost) {
  return guarded(ctx, [&]() { return impl_inflate(ctx, lethals, n, invalid, params, out_dist, out_cost); });
}
int32_t mnb_inflation_update(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid,
                             const mnb_inflation_params* params, float* out_dist, float* out_cost, uint32_t* out_changed,
                             uint32_t* n_changed) {
  return guarded(ctx, [&]() { return impl_inflation_update(ctx, lethals, n, invalid, params, out_dist, out_cost, out_changed, n_changed); });
}
int32_t mnb_compute_layers(mnb_ctx* ctx, const mnb_layer_params* params, const float* clearance, float* out_costs,
                           float* out_combined, uint8_t* out_lethal_mask) {
  return guarded(ctx, [&]() { return impl_compute_layers(ctx, params, clearance, out_costs, out_combined, out_lethal_mask); });
}
int32_t mnb_set_costs(mnb_ctx* ctx, const float* vertex_costs, const float* edge_weights, const uint8_t* invalid) {
  return guarded(ctx, [&]() { return impl_set_costs(ctx, vertex_costs, edge_weights, invalid); });
}
int32_t mnb_compute_edge_weights(mnb_ctx* ctx, const float* vertex_costs, double edge_cost_factor, float* out_w) {
  return guarded(ctx, [&]() { return impl_compute_edge_weights(ctx, vertex_costs, edge_cost_factor, out_w); });
}
int32_t mnb_locate(mnb_ctx* ctx, uint32_t n, const float* points, uint32_t* out_vertex, int32_t* out_face, float* out_bary) {
  return guarded(ctx, [&]() { return impl_locate(ctx, n, points, out_vertex, out_face, out_bary); });
}
int32_t mnb_vector_map(mnb_ctx* ctx, const uint32_t* pred, const float* direction, const int32_t* cutting_face, float* out_vec) {
  return guarded(ctx, [&]() { return impl_vector_map(ctx, pred, direction, cutting_face, out_vec); });
}
int32_t mnb_inflation_vector_map(mnb_ctx* ctx, float* out_vectors) {
  return guarded(ctx, [&]() { return impl_inflation_vector_map(ctx, out_vectors); });
}
int32_t mnb_inflation_vector_at(mnb_ctx* ctx, uint32_t n, const uint32_t* faces_q, const float* bary, float* out) {
  return guarded(ctx, [&]() { return impl_inflation_vector_at(ctx, n, faces_q, bary, out); });
}
int32_t mnb_cvp_backtrack(mnb_ctx* ctx, const float robot_pos[3], uint32_t robot_face, double step_width, uint32_t max_points,
                          float* path_pos, uint32_t* path_face, uint32_t* n_points) {
  return guarded(ctx, [&]() { return impl_cvp_backtrack(ctx, robot_pos, robot_face, step_width, max_points, path_pos, path_face, n_points); });
}
int32_t mnb_update_vertex_costs(mnb_ctx* ctx, uint32_t n_changed, const uint32_t* changed, const float* costs,
                                int32_t costs_indexed_by_vertex, float default_value, double edge_cost_factor) {
  return guarded(ctx, [&]() { return impl_update_vertex_costs(ctx, n_changed, changed, costs, costs_indexed_by_vertex, default_value, edge_cost_factor); });
}
int32_t mnb_max_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const uint8_t* const* layer_lethal, uint32_t n_changed, const uint32_t* changed,
                                   float* io_costs, uint8_t* io_lethal) {
  return guarded(ctx, [&]() { return impl_max_combination_update(ctx, n_layers, layer_costs, defaults, layer_lethal, n_changed, changed, io_costs, io_lethal); });
}
int32_t mnb_avg_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const float* weights, const uint8_t* const* layer_lethal, uint32_t n_changed,
                                   const uint32_t* changed, float* io_costs, uint8_t* io_lethal) {
  return guarded(ctx, [&]() { return impl_avg_combination_update(ctx, n_layers, layer_costs, defaults, weights, layer_lethal, n_changed, changed, io_costs, io_lethal); });
}

}  // extern "C"

#include "raycast_host.cuh"
#include "group.cuh"
