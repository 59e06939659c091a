// Multi-GPU entry points of the C ABI (SURVEY.md 8e): one host process drives N devices, every device holds a replica of
// the map, goal k of a batch belongs to rank k mod N, and the potential fields are all-gathered over NCCL (NVLink /
// NVSwitch) into every device.  The wavefront itself never leaves its device -- the path shards across queries and not
// inside one -- so the gather is the only collective and there is no compute step to fuse it with.
// (part of libmeshnav_b200.so: included by meshnav.cu after the single-device entry points)
//
// NCCL is bound at run time (dlopen of libnccl.so.2, the one the process already has if torch loaded it): the
// single-device library has no link-time dependency on it, and a group of ONE device never touches it.
#pragma once
#include <dlfcn.h>
#include <thread>

namespace mnbg {
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;
struct Nccl {
  void* handle = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int /*ncclDataType_t*/, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string& err) {
    if (handle) return true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) { handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (handle) break; }
    if (!handle) { err = std::string("NCCL not found: ") + dlerror(); return false; }
    auto sym = [&](const char* n) { return dlsym(handle, n); };
    CommInitAll = (decltype(CommInitAll))sym("ncclCommInitAll"); CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
    AllGather = (decltype(AllGather))sym("ncclAllGather"); GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd"); GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
    if (!CommInitAll || !CommDestroy || !AllGather || !GroupStart || !GroupEnd) { err = "NCCL symbols missing"; return false; }
    return true;
  }
};
constexpr int NCCL_UINT32 = 3;    // ncclUint32  (nccl.h: ncclDataType_t)
constexpr int NCCL_FLOAT32 = 7;   // ncclFloat32
}  // namespace mnbg

struct mnb_group {
  std::vector<mnb_ctx*> ctx;
  std::vector<mnbg::ncclComm_t> comm;
  std::vector<float*> d_fields;         // per device: [N][pad][V] gathered potentials (library-owned, grows on demand)
  std::vector<size_t> cap;
  std::vector<uint32_t*> d_preds;       // per device: [N][pad][V] predecessors of the last Dijkstra batch with want_pred
  std::vector<size_t> pred_cap;
  mnbg::Nccl nccl;
  std::string err;
  uint32_t last_n = 0, last_pad = 0;
  bool last_has_pred = false;           // the last sharded call was mnb_dijkstra_batch_sharded with want_pred
};

extern "C" {

// one context per device (devices[i] = CUDA ordinal) + the communicators of the gather
int32_t mnb_group_create(int32_t n_devices, const int32_t* devices, mnb_group** out_group) {
  if (!out_group || n_devices <= 0 || !devices) return MNB_E_ARG;
  *out_group = nullptr;
  mnb_group* g = new mnb_group();
  int32_t rc = MNB_OK;
  for (int32_t i = 0; i < n_devices && rc == MNB_OK; ++i) { mnb_ctx* c = nullptr; rc = mnb_create(devices[i], &c); if (rc == MNB_OK) g->ctx.push_back(c); }
  if (rc == MNB_OK && n_devices > 1) {
    if (!g->nccl.load(g->err)) rc = MNB_E_NCCL;
    else {
      g->comm.resize((size_t)n_devices);
      std::vector<int> devs(devices, devices + n_devices);
      if (g->nccl.CommInitAll(g->comm.data(), n_devices, devs.data()) != 0) { g->comm.clear(); rc = MNB_E_NCCL; }
    }
  }
  if (rc != MNB_OK) { for (mnb_ctx* c : g->ctx) mnb_destroy(c); delete g; return rc; }
  g->d_fields.assign((size_t)n_devices, nullptr); g->cap.assign((size_t)n_devices, 0);
  g->d_preds.assign((size_t)n_devices, nullptr); g->pred_cap.assign((size_t)n_devices, 0);
  *out_group = g;
  return MNB_OK;
}

void mnb_group_destroy(mnb_group* g) {
  if (!g) return;
  for (size_t r = 0; r < g->ctx.size(); ++r) {
    cudaSetDevice(g->ctx[r]->device);
    if (g->d_fields[r]) cudaFree(g->d_fields[r]);
    if (g->d_preds[r]) cudaFree(g->d_preds[r]);
    if (r < g->comm.size() && g->comm[r]) g->nccl.CommDestroy(g->comm[r]);
    mnb_destroy(g->ctx[r]);
  }
  delete g;
}

int32_t mnb_group_size(mnb_group* g) { return g ? (int32_t)g->ctx.size() : 0; }
mnb_ctx* mnb_group_ctx(mnb_group* g, int32_t rank) { return (g && rank >= 0 && (size_t)rank < g->ctx.size()) ? g->ctx[(size_t)rank] : nullptr; }
const char* mnb_group_last_error(mnb_group* g) { return g ? g->err.c_str() : "null group"; }

// the map and the per-plan costs are replicated on every device (HOST pointers; the devices upload concurrently)
static int32_t group_foreach(mnb_group* g, const std::function<int32_t(mnb_ctx*, size_t)>& f) {
  std::vector<int32_t> rc(g->ctx.size(), MNB_OK);
  std::vector<std::thread> th;
  for (size_t r = 0; r < g->ctx.size(); ++r) th.emplace_back([&, r]() { rc[r] = f(g->ctx[r], r); });
  for (auto& t : th) t.join();
  for (size_t r = 0; r < rc.size(); ++r) if (rc[r] != MNB_OK) { g->err = "rank " + std::to_string(r) + ": " + g->ctx[r]->err; return rc[r]; }
  return MNB_OK;
}
int32_t mnb_group_set_mesh(mnb_group* g, uint32_t V, uint32_t F, const float* pos, const uint32_t* faces, const uint32_t* edges, uint32_t E) {
  if (!g) return MNB_E_ARG;
  return group_foreach(g, [&](mnb_ctx* c, size_t) { return mnb_set_mesh(c, V, F, pos, faces, edges, E); });
}
int32_t mnb_group_set_costs(mnb_group* g, const float* vertex_costs, const float* edge_weights, const uint8_t* invalid) {
  if (!g) return MNB_E_ARG;
  return group_foreach(g, [&](mnb_ctx* c, size_t) { if (c->ptr_mode != MNB_PTR_HOST) return (int32_t)MNB_E_STATE; return mnb_set_costs(c, vertex_costs, edge_weights, invalid); });
}

// MeshMap::layerChanged on every replica (mnb_update_vertex_costs per device, concurrently): keeps the maps of a group in step
// under dynamic obstacles without re-uploading V + E floats per device.  HOST arrays.
int32_t mnb_group_update_vertex_costs(mnb_group* g, uint32_t n_changed, const uint32_t* changed, const float* costs,
                                      int32_t costs_indexed_by_vertex, float default_value, double edge_cost_factor) {
  if (!g) return MNB_E_ARG;
  return group_foreach(g, [&](mnb_ctx* c, size_t) {
    if (c->ptr_mode != MNB_PTR_HOST) return (int32_t)MNB_E_STATE;
    return mnb_update_vertex_costs(c, n_changed, changed, costs, costs_indexed_by_vertex, default_value, edge_cost_factor);
  });
}

// grows the per-device [N][pad][V] buffers of a sharded call to hold `need` elements
extern "C++" {
template <class T>
static int32_t group_grow(mnb_group* g, std::vector<T*>& buf, std::vector<size_t>& cap, size_t need) {
  for (size_t r = 0; r < g->ctx.size(); ++r) {
    if (cap[r] >= need) continue;
    cudaSetDevice(g->ctx[r]->device);
    if (buf[r]) cudaFree(buf[r]);
    buf[r] = nullptr; cap[r] = 0;
    if (cudaMalloc((void**)&buf[r], need * sizeof(T)) != cudaSuccess) { g->err = "gather buffer: out of device memory"; return MNB_E_NOMEM; }
    cap[r] = need;
  }
  return MNB_OK;
}
}  // extern "C++"

// in-place all-gather of every rank's slot of the fields (and, with preds, of the predecessors) in one NCCL group call
static int32_t group_gather(mnb_group* g, size_t slot, bool preds) {
  const size_t N = g->ctx.size();
  if (g->nccl.GroupStart() != 0) { g->err = "ncclGroupStart"; return MNB_E_NCCL; }
  for (size_t r = 0; r < N; ++r) {
    int e = g->nccl.AllGather(g->d_fields[r] + r * slot, g->d_fields[r], slot, mnbg::NCCL_FLOAT32, g->comm[r], g->ctx[r]->stream);
    if (e == 0 && preds) e = g->nccl.AllGather(g->d_preds[r] + r * slot, g->d_preds[r], slot, mnbg::NCCL_UINT32, g->comm[r], g->ctx[r]->stream);
    if (e != 0) { g->nccl.GroupEnd(); g->err = std::string("ncclAllGather: ") + (g->nccl.GetErrorString ? g->nccl.GetErrorString(e) : "?"); return MNB_E_NCCL; }
  }
  if (g->nccl.GroupEnd() != 0) { g->err = "ncclGroupEnd"; return MNB_E_NCCL; }
  for (size_t r = 0; r < N; ++r) { cudaSetDevice(g->ctx[r]->device); if (cudaStreamSynchronize(g->ctx[r]->stream) != cudaSuccess) { g->err = "gather: stream sync failed"; return MNB_E_CUDA; } }
  return MNB_OK;
}

// Batched full-field CVP plans, sharded: goal k -> rank k mod N.  Every rank plans its goals (mnb_cvp_batch on its device,
// all devices concurrently) straight into its slot of the gather buffer; one in-place ncclAllGather then leaves ALL fields
// on EVERY device.  Layout of the per-device result (library-owned device memory, valid until the next sharded call):
// float[N][pad][V] with pad = ceil(n / N); the field of goal k is row mnb_group_row(group, k) = (k mod N) * pad + k / N.
// gather = 0 skips the collective (each device then only holds its own shard's rows).
int32_t mnb_cvp_batch_sharded(mnb_group* g, uint32_t n, const uint32_t* seed_faces, const float* seed_pos, double cost_limit, int32_t gather) {
  if (!g || n == 0 || !seed_faces || !seed_pos) return MNB_E_ARG;
  const uint32_t N = (uint32_t)g->ctx.size(), pad = (n + N - 1) / N;
  const size_t V = g->ctx[0]->V;
  if (!V) { g->err = "mnb_group_set_mesh / mnb_group_set_costs not called"; return MNB_E_STATE; }
  g->last_has_pred = false;
  int32_t rc = group_grow(g, g->d_fields, g->cap, (size_t)N * pad * V);
  if (rc != MNB_OK) return rc;
  rc = group_foreach(g, [&](mnb_ctx* c, size_t r) -> int32_t {
    std::vector<uint32_t> sf; std::vector<float> sp;
    for (uint32_t k = (uint32_t)r; k < n; k += N) { sf.push_back(seed_faces[k]); sp.insert(sp.end(), seed_pos + 3 * (size_t)k, seed_pos + 3 * (size_t)k + 3); }
    if (sf.empty()) return MNB_OK;
    const int old_mode = c->ptr_mode;
    c->ptr_mode = MNB_PTR_DEVICE;        // (only the output is a device pointer: seeds are always host arrays)
    const int32_t b = mnb_cvp_batch(c, (uint32_t)sf.size(), sf.data(), sp.data(), cost_limit, g->d_fields[r] + r * (size_t)pad * V);
    c->ptr_mode = old_mode;
    return b;
  });
  if (rc != MNB_OK) return rc;
  g->last_n = n; g->last_pad = pad;
  if (gather && N > 1 && (rc = group_gather(g, (size_t)pad * V, false)) != MNB_OK) return rc;
  return MNB_SUCCESS;
}

// Batched full-field Dijkstra plans, sharded the same way (mnb_dijkstra_batch per rank): distances into the fields buffers
// above, with want_pred the predecessors into d_preds in the same layout; both are gathered in one NCCL group call.
int32_t mnb_dijkstra_batch_sharded(mnb_group* g, uint32_t n, const uint32_t* seed_vertices, double cost_limit, int32_t want_pred, int32_t gather) {
  if (!g || n == 0 || !seed_vertices) return MNB_E_ARG;
  const uint32_t N = (uint32_t)g->ctx.size(), pad = (n + N - 1) / N;
  const size_t V = g->ctx[0]->V;
  if (!V) { g->err = "mnb_group_set_mesh / mnb_group_set_costs not called"; return MNB_E_STATE; }
  g->last_has_pred = false;
  int32_t rc = group_grow(g, g->d_fields, g->cap, (size_t)N * pad * V);
  if (rc == MNB_OK && want_pred) rc = group_grow(g, g->d_preds, g->pred_cap, (size_t)N * pad * V);
  if (rc != MNB_OK) return rc;
  rc = group_foreach(g, [&](mnb_ctx* c, size_t r) -> int32_t {
    std::vector<uint32_t> sv;
    for (uint32_t k = (uint32_t)r; k < n; k += N) sv.push_back(seed_vertices[k]);
    if (sv.empty()) return MNB_OK;
    const int old_mode = c->ptr_mode;
    c->ptr_mode = MNB_PTR_DEVICE;        // (only the outputs are device pointers: seeds are always host arrays)
    const size_t off = r * (size_t)pad * V;
    const int32_t b = mnb_dijkstra_batch(c, (uint32_t)sv.size(), sv.data(), cost_limit, g->d_fields[r] + off, want_pred ? g->d_preds[r] + off : nullptr);
    c->ptr_mode = old_mode;
    return b;
  });
  if (rc != MNB_OK) return rc;
  g->last_n = n; g->last_pad = pad; g->last_has_pred = want_pred != 0;
  if (gather && N > 1 && (rc = group_gather(g, (size_t)pad * V, want_pred != 0)) != MNB_OK) return rc;
  return MNB_SUCCESS;
}

uint32_t mnb_group_row(mnb_group* g, uint32_t goal) { if (!g || !g->last_pad) return 0; const uint32_t N = (uint32_t)g->ctx.size(); return (goal % N) * g->last_pad + goal / N; }
// device pointer of the gathered fields on `rank` (float[N][pad][V], see mnb_cvp_batch_sharded)
float* mnb_group_fields(mnb_group* g, int32_t rank) { return (g && rank >= 0 && (size_t)rank < g->ctx.size()) ? g->d_fields[(size_t)rank] : nullptr; }
// copies the fields of goals [first, first + count) from `rank`'s buffer into host memory, in goal order
int32_t mnb_group_read_fields(mnb_group* g, int32_t rank, uint32_t first, uint32_t count, float* out_host) {
  if (!g || rank < 0 || (size_t)rank >= g->ctx.size() || !out_host || first + count > g->last_n) return MNB_E_ARG;
  mnb_ctx* c = g->ctx[(size_t)rank];
  const size_t V = c->V;
  if (cudaSetDevice(c->device) != cudaSuccess) return MNB_E_CUDA;
  for (uint32_t k = 0; k < count; ++k)
    if (cudaMemcpyAsync(out_host + (size_t)k * V, g->d_fields[(size_t)rank] + (size_t)mnb_group_row(g, first + k) * V, sizeof(float) * V, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return MNB_E_CUDA;
  return cudaStreamSynchronize(c->stream) == cudaSuccess ? MNB_OK : MNB_E_CUDA;
}

// device pointer of the predecessors on `rank` (uint32[N][pad][V], see mnb_dijkstra_batch_sharded)
uint32_t* mnb_group_preds(mnb_group* g, int32_t rank) { return (g && rank >= 0 && (size_t)rank < g->ctx.size()) ? g->d_preds[(size_t)rank] : nullptr; }
// copies the predecessors of goals [first, first + count) from `rank`'s buffer into host memory, in goal order
int32_t mnb_group_read_preds(mnb_group* g, int32_t rank, uint32_t first, uint32_t count, uint32_t* out_host) {
  if (!g || rank < 0 || (size_t)rank >= g->ctx.size() || !out_host || first + count > g->last_n) return MNB_E_ARG;
  if (!g->last_has_pred) { g->err = "mnb_group_read_preds needs a preceding mnb_dijkstra_batch_sharded with want_pred"; return MNB_E_STATE; }
  mnb_ctx* c = g->ctx[(size_t)rank];
  const size_t V = c->V;
  if (cudaSetDevice(c->device) != cudaSuccess) return MNB_E_CUDA;
  for (uint32_t k = 0; k < count; ++k)
    if (cudaMemcpyAsync(out_host + (size_t)k * V, g->d_preds[(size_t)rank] + (size_t)mnb_group_row(g, first + k) * V, sizeof(uint32_t) * V, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return MNB_E_CUDA;
  return cudaStreamSynchronize(c->stream) == cudaSuccess ? MNB_OK : MNB_E_CUDA;
}

}  // extern "C"
