/*
 * meshnav_b200.h -- C ABI of libmeshnav_b200.so
 *
 * B200-native (sm_100a CUDA) replacement for the wavefront hot path of
 * naturerobots/mesh_navigation.  Plain pointers and sizes only; no C++ / torch
 * types cross this boundary.  Every entry point names the reference interface
 * it stands in for (paths relative to the reference repo).
 *
 * Conventions
 *   - all calls return MNB_OK (0) or a negative MNB_E_* code, except the
 *     planner calls which return the MBF GetPath::Result code the reference's
 *     makePlan would return (dijkstra_mesh_planner.h:72-85): 0 SUCCESS,
 *     51 CANCELED, 52 INVALID_START, 53 INVALID_GOAL, 54 NO_PATH_FOUND,
 *     or a negative MNB_E_* code on CUDA / argument errors.
 *   - array arguments are HOST pointers by default.  After
 *     mnb_set_pointer_mode(ctx, MNB_PTR_DEVICE) array arguments of the
 *     per-call functions (costs, weights, outputs) are DEVICE pointers on the
 *     context's device and no host<->device copy happens inside the call.
 *   - the library never frees or keeps caller memory; outputs are written into
 *     caller-provided buffers of the stated length.
 *   - an mnb_ctx is single-caller (one stream); mnb_cancel() is the only entry
 *     point that may be called concurrently from another thread
 *     (reference: CVPMeshPlanner::cancel, cvp_mesh_planner.cpp:142-146).
 *   - there is NO CPU fallback: every compute entry point fails with
 *     MNB_E_CUDA if no sm_100 device is usable.
 */
#ifndef MESHNAV_B200_H
#define MESHNAV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MNB_OK 0
#define MNB_E_ARG (-1)
#define MNB_E_CUDA (-2)
#define MNB_E_STATE (-3)
#define MNB_E_NCCL (-4)
#define MNB_E_NOMEM (-5)

/* MBF outcome codes (mbf_msgs/action/GetPath; dijkstra_mesh_planner.h:72-85) */
#define MNB_SUCCESS 0
#define MNB_CANCELED 51
#define MNB_INVALID_START 52
#define MNB_INVALID_GOAL 53
#define MNB_NO_PATH_FOUND 54

#define MNB_PTR_HOST 0
#define MNB_PTR_DEVICE 1

typedef struct mnb_ctx mnb_ctx;

/* ---- lifetime ----------------------------------------------------------- */
int32_t mnb_create(int32_t device, mnb_ctx** out_ctx);
void mnb_destroy(mnb_ctx* ctx);
const char* mnb_last_error(mnb_ctx* ctx);
int32_t mnb_set_pointer_mode(mnb_ctx* ctx, int32_t mode);
/* cudaStream_t (as void*) the context launches on; lets a caller time with CUDA events. */
void* mnb_stream(mnb_ctx* ctx);

/* ---- map upload: replaces the lvr2 half-edge mesh the plugins read ------
 * mesh_map::MeshMap::mesh() / edgeDistances() (mesh_map.h:97-452, mesh_map.cpp:404-425).
 * pos[3V] float xyz, faces[3F] vertex ids in the mesh's cyclic (CCW) order.
 * edges[2E] may be NULL: the library then numbers edges by ascending (lo,hi)
 * vertex pair; pass the caller's own edge order (e.g. lvr2 EdgeHandle order)
 * so that edge_weights / edge_distances arrays use the caller's indices.
 * Always HOST pointers (one-time setup). */
int32_t mnb_set_mesh(mnb_ctx* ctx, uint32_t V, uint32_t F, const float* pos, const uint32_t* faces,
                     const uint32_t* edges, uint32_t E);
uint32_t mnb_num_vertices(mnb_ctx* ctx);
uint32_t mnb_num_faces(mnb_ctx* ctx);
uint32_t mnb_num_edges(mnb_ctx* ctx);
int32_t mnb_get_edges(mnb_ctx* ctx, uint32_t* out_edges /* 2E, host */);
/* lvr2::calcVertexDistances as used for MeshMap::edge_distances (mesh_map.cpp:414) */
int32_t mnb_get_edge_distances(mnb_ctx* ctx, float* out_edge_distances /* E */);

/* ---- MeshMap::computeEdgeWeights (mesh_map.cpp:517-561) -----------------
 * edge_weights[e] = +inf if an endpoint cost is inf, else
 * dist[e] + edge_cost_factor * (dist[e] * (c1 + c2) / 2).  Writes out_edge_weights (E) if
 * non-NULL and installs vertex_costs + the weights as the planners' inputs. */
int32_t mnb_compute_edge_weights(mnb_ctx* ctx, const float* vertex_costs /* V */, double edge_cost_factor,
                                 float* out_edge_weights /* E or NULL */);

/* ---- per-plan inputs the planners read from the map ---------------------
 * MeshMap::vertexCosts() / edgeWeights() / invalid
 * (cvp_mesh_planner.cpp:245,663-664; dijkstra_mesh_planner.cpp:214,227-229).
 * invalid may be NULL (no invalid vertices). */
int32_t mnb_set_costs(mnb_ctx* ctx, const float* vertex_costs /* V */, const float* edge_weights /* E */,
                      const uint8_t* invalid /* V or NULL */);

/* ---- DijkstraMeshPlanner::dijkstra (dijkstra_mesh_planner.cpp:217-398) ---
 * seed_vertex  = the reference's start_vertex (nearest vertex to the navigation goal, :235)
 * robot_vertex = the reference's goal_vertex (nearest vertex to the robot, :236) or -1 for a
 *                full field.  out_dist[V] (+inf = unreached), out_pred[V] (self = none). */
int32_t mnb_dijkstra(mnb_ctx* ctx, uint32_t seed_vertex, int64_t robot_vertex, double cost_limit,
                     double goal_dist_offset, float* out_dist, uint32_t* out_pred);

/* ---- CVPMeshPlanner::waveFrontPropagation (cvp_mesh_planner.cpp:651-886) -
 * seed_face / seed_pos = the reference's start_face / start (navigation goal, :673,:719-728)
 * robot_face           = the reference's goal_face (:674) or -1 for a full field.
 * Outputs (any may be NULL): potential_ , predecessors_, direction_, cutting_faces_ (-1 = none). */
int32_t mnb_cvp(mnb_ctx* ctx, uint32_t seed_face, const float seed_pos[3], int64_t robot_face,
                double cost_limit, double goal_dist_offset, float* out_dist, uint32_t* out_pred,
                float* out_direction, int32_t* out_cutting_face);

/* Batched full-field CVP potentials: n independent goals on the installed map, one wavefront
 * per thread-block cluster, all SMs busy.  out_dist is [n][V] row-major. */
int32_t mnb_cvp_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_faces /* n, host */,
                      const float* seed_pos /* 3n, host */, double cost_limit, float* out_dist);

/* Batched full-field Dijkstra: n independent DijkstraMeshPlanner::dijkstra runs (robot_vertex = -1) on the installed map,
 * one goal per thread block (or cluster), all SMs busy.  Row k of out_dist / out_pred is bit for bit what
 * mnb_dijkstra(ctx, seed_vertices[k], -1, cost_limit, ...) writes.  out_dist [n][V] (+inf = unreached), out_pred [n][V]
 * or NULL (self = none).  Edge weights must be >= 0.  Duplicate seeds are allowed; an invalid seed is still expanded.
 * MNB_INVALID_START (nothing written) if a seed is >= V.  Leaves the result of the last mnb_cvp (mnb_cvp_backtrack,
 * mnb_vector_map(pred = NULL)) untouched. */
int32_t mnb_dijkstra_batch(mnb_ctx* ctx, uint32_t n, const uint32_t* seed_vertices /* n, host */, double cost_limit,
                           float* out_dist, uint32_t* out_pred);

/* ---- InflationLayer::waveCostInflation (inflation_layer.cpp:341-491) -----
 * lethals[n] (any order, duplicates allowed).  Uses edge_distances (:383), not edge_weights.
 * out_dist[V]: distances_ (+inf = not in the sparse map); out_cost[V]: riskiness_ =
 * fading(dist) (NaN = not in the sparse map).  Either may be NULL. */
typedef struct mnb_inflation_params {
  double inscribed_radius;    /* 0.25  (inflation_layer.h:240-248) */
  double inflation_radius;    /* 0.4  */
  double lethal_value;        /* 1.0  */
  double inscribed_value;     /* 0.99 */
  double cost_scaling_factor; /* 1.0  */
} mnb_inflation_params;
int32_t mnb_inflate(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid /* V or NULL */,
                    const mnb_inflation_params* params, float* out_dist, float* out_cost);

/* ---- geometric cost layers + MaxCombinationLayer (mesh_layers/src/<name>_layer.cpp) -------------------
 * HeightDiffLayer::computeLayer (height_diff_layer.cpp:103-110), RoughnessLayer (roughness_layer.cpp:91-147),
 * SteepnessLayer (steepness_layer.cpp:100-170), RidgeLayer (ridge_layer.cpp:101-187), ClearanceLayer cost
 * mapping (clearance_layer.cpp:67-99, on a caller-provided clearance array; NULL = +inf, no ray hits),
 * BorderLayer (border_layer.cpp:104-110), computeLethals (cost > threshold) and
 * MaxCombinationLayer::computeLayer (combination_layer.cpp:44-85), fused into ONE per-vertex kernel.
 * out_costs: 6*V floats, layer-major in the order height_diff, roughness, steepness, ridge, clearance,
 * border; out_combined: V; out_lethal_mask: V bytes, bit i = lethal in layer i.  Any output may be NULL;
 * the results also stay resident on the device for chaining. */
typedef struct mnb_layer_params {
  double height_diff_threshold, height_diff_radius;           /* 0.185, 0.3 */
  double roughness_threshold, roughness_radius;               /* 0.3, 0.3 */
  double steepness_threshold;                                 /* 0.3 */
  double ridge_threshold, ridge_radius;                       /* 0.3, 0.3 */
  double clearance_robot_height, clearance_height_inflation;  /* 0.5, 0.3 */
  double border_threshold, border_cost;                       /* 0.5, 1.0 */
} mnb_layer_params;
int32_t mnb_compute_layers(mnb_ctx* ctx, const mnb_layer_params* params, const float* clearance /* V or NULL */,
                           float* out_costs, float* out_combined, uint8_t* out_lethal_mask);
/* lvr2::calcVertexNormals equivalent (mesh_map.cpp:374): normalised sum of incident face normals */
int32_t mnb_get_vertex_normals(mnb_ctx* ctx, float* out_normals /* 3V */);

/* ---- localisation -----------------------------------------------------------------------------------
 * MeshMap::getNearestVertexHandle (mesh_map.cpp:1161-1174) and MeshMap::searchContainingFace / getContainingFace
 * (mesh_map.cpp:1110-1159) for n query points at once: out_vertex[q] = nearest vertex (exhaustive, ties to the lowest
 * id), out_face[q] = the incident face of that vertex containing the projected point (-1: none), out_bary its
 * barycentric coordinates.  Any of the outputs may be NULL. */
int32_t mnb_locate(mnb_ctx* ctx, uint32_t n, const float* points /* 3n */, uint32_t* out_vertex /* n */,
                   int32_t* out_face /* n */, float* out_bary /* 3n */);

/* ---- vector-field epilogues -----------------------------------------------------------------------
 * DijkstraMeshPlanner::computeVectorMap (dijkstra_mesh_planner.cpp:189-209): direction == NULL, cutting_face == NULL:
 *   out[v] = normalize(p[pred[v]] - p[v]).
 * CVPMeshPlanner::computeVectorMap (cvp_mesh_planner.cpp:204-239): the vector is additionally rotated about the vertex
 *   normal by direction[v]; vertices without a cutting face are skipped.
 * out_vec: 3V floats, NaN = "no entry in the sparse vector map" (pred[v] == v or no cutting face).
 * pred == NULL: the field of the LAST successful mnb_cvp on this context, from its device-resident result (nothing is uploaded). */
int32_t mnb_vector_map(mnb_ctx* ctx, const uint32_t* pred /* V or NULL */, const float* direction /* V or NULL */,
                       const int32_t* cutting_face /* V or NULL */, float* out_vec /* 3V */);

/* ---- vector-field back-tracking -------------------------------------------------------------------
 * The tail of CVPMeshPlanner::waveFrontPropagation (cvp_mesh_planner.cpp:920-951): follows the vector field of the
 * LAST successful mnb_cvp on this context (kept on the device) from the robot position down to the wave's seed with
 * MeshMap::meshAhead (mesh_map.cpp:1070-1108) in steps of step_width.  Points are returned in walk order
 * (robot first, seed last = the order of the final plan after cvp:100 path.reverse()).  In device-pointer mode
 * the result arrays of that mnb_cvp must still be alive.  Layer vector fields (AbstractLayer::vectorAt) are zero.
 * Returns MNB_SUCCESS / MNB_NO_PATH_FOUND / MNB_CANCELED; MNB_E_STATE if max_points is exhausted. */
int32_t mnb_cvp_backtrack(mnb_ctx* ctx, const float robot_pos[3], uint32_t robot_face, double step_width, uint32_t max_points,
                          float* path_pos /* 3*max_points */, uint32_t* path_face /* max_points or NULL */,
                          uint32_t* n_points);

/* ---- incremental updates: the sensor-rate callers of the hot path (SURVEY.md 3.4) ----------------------------------
 * NaN marks "no entry" in a sparse lvr2 cost map; `changed` plays the std::set<VertexHandle> of the reference
 * (any order, duplicates allowed).  All three work on the changed vertices only. */

/* MeshMap::layerChanged (mesh_map.cpp:455-492) + MeshMap::updateEdgeWeights (mesh_map.cpp:563-618):
 *   vertex_costs[v] = cost_map.get(v).value_or(default_value) for v in changed, then the weights of the edges incident
 *   to a changed vertex are recomputed with the formula of computeEdgeWeights -- and, exactly as in the reference
 *   (:568-572), NOT AT ALL when edge_cost_factor == 0.  The planners' derived tables are refreshed for those edges only
 *   (no V- or E-sized pass, no re-upload).  costs_indexed_by_vertex == 0: costs[i] is the new cost of changed[i];
 *   != 0: costs is the layer's V-sized map and default_value replaces NaN entries.  Needs mnb_set_costs /
 *   mnb_compute_edge_weights first. */
int32_t mnb_update_vertex_costs(mnb_ctx* ctx, uint32_t n_changed, const uint32_t* changed, const float* costs,
                                int32_t costs_indexed_by_vertex, float default_value, double edge_cost_factor);
/* the installed per-plan inputs (MeshMap::vertexCosts() / edgeWeights()); either may be NULL */
int32_t mnb_get_costs(mnb_ctx* ctx, float* out_vertex_costs /* V */, float* out_edge_weights /* E */);

/* MaxCombinationLayer::onInputChanged (combination_layer.cpp:87-147) for the changed vertices:
 *   io_costs[v] = max(0, max_i (layer_costs[i][v] or defaults[i]));  io_lethal[v] = OR_i layer_lethal[i][v].
 * layer_costs / layer_lethal are HOST arrays of n_layers (<= 8) pointers to V-sized maps (host or device per the
 * pointer mode); layer_lethal, any of its entries and io_lethal may be NULL; defaults is a host array. */
int32_t mnb_max_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const uint8_t* const* layer_lethal, uint32_t n_changed, const uint32_t* changed,
                                   float* io_costs /* V */, uint8_t* io_lethal /* V or NULL */);

/* AvgCombinationLayer::onInputChanged / computeLayer (combination_layer.cpp:185-302) for the changed vertices:
 *   io_costs[v] = sum_i weights[i] * (layer_costs[i][v] or defaults[i]), accumulated in layer order in float;
 *   io_lethal[v] = OR_i layer_lethal[i][v].  weights = AbstractLayer::combinationWeight() of the inputs (host array). */
int32_t mnb_avg_combination_update(mnb_ctx* ctx, uint32_t n_layers, const float* const* layer_costs, const float* defaults,
                                   const float* weights, const uint8_t* const* layer_lethal, uint32_t n_changed,
                                   const uint32_t* changed, float* io_costs /* V */, uint8_t* io_lethal /* V or NULL */);

/* InflationLayer::onInputChanged (inflation_layer.cpp:97-179): re-runs waveCostInflation from `lethals` (the reference
 * does a full re-inflation here too, :143-151) and reports the update set handed to notifyChange (:154-176): the
 * vertices that carry a riskiness value now or carried one after the previous mnb_inflate / mnb_inflation_update on this
 * context, ascending.  out_changed: room for V ids (may be NULL); *n_changed (host) receives the count. */
int32_t mnb_inflation_update(mnb_ctx* ctx, const uint32_t* lethals, uint32_t n, const uint8_t* invalid /* V or NULL */,
                             const mnb_inflation_params* params, float* out_dist, float* out_cost,
                             uint32_t* out_changed /* V */, uint32_t* n_changed);

/* ---- ray casting against the map -------------------------------------------------------------------------------------
 * The shared raycaster of the map (MeshMap::raycaster(), mesh_map.h:318; lvr2::EmbreeRaycaster / BVHRaycaster built at
 * mesh_map.cpp:317-321) as a linear BVH over the faces on the device, built at the first ray call after mnb_set_mesh.
 * Results are those of a loop over all faces (the tree only prunes): two-sided Moeller-Trumbore in float, nearest hit,
 * ties to the smallest face id -- the arithmetic is spelled out in oracle/oracle.cpp ("Ray casting against the map").
 *
 * mnb_cast_rays = RaycasterBase::castRays as called at obstacle_layer.cpp:239.  dirs: one unit vector per ray
 * (dir_stride 3) or one for all rays (dir_stride 0, obstacle_layer.cpp:229).  Outputs (each may be NULL): hit flag,
 * distance (+inf: no hit), face id (0xffffffff: no hit), hit point (NaN: no hit). */
int32_t mnb_cast_rays(mnb_ctx* ctx, uint32_t n, const float* origins /* 3n */, const float* dirs, uint32_t dir_stride,
                      uint8_t* out_hit /* n */, float* out_dist /* n */, uint32_t* out_face /* n */, float* out_point /* 3n */);

/* ObstacleLayer::processPointCloud (obstacle_layer.cpp:215-296) without the ROS plumbing: points are the cloud in the
 * message frame; tf the row-major 3x4 [R|t] of the message frame -> map frame transform (:176-180); down_axis the
 * configured axis already rotated into the map frame (:183-205).  Points with |p| <= max_obstacle_dist are transformed
 * and cast along down_axis; a hit within robot_height makes the three vertices of the hit face lethal (:245-256).
 * out_lethals: the new lethal set, ascending (lethals_); out_changed: its symmetric difference with the set of the
 * previous call on this context (:268-273, what notifyChange receives); both need room for V ids and may be NULL; the
 * counts go to the host.  out_costs (V floats or NULL): +inf on lethal vertices, NaN = no entry (costs_, :250;
 * defaultValue() 0).  mnb_obstacle_reset empties the remembered lethal set. */
typedef struct mnb_obstacle_params {
  double max_obstacle_dist, robot_height;
  float tf[12];
  float down_axis[3];
} mnb_obstacle_params;
int32_t mnb_obstacle_update(mnb_ctx* ctx, uint32_t n_points, const float* points /* 3n */, const mnb_obstacle_params* params,
                            uint32_t* out_lethals /* V */, uint32_t* n_lethals, uint32_t* out_changed /* V */,
                            uint32_t* n_changed, float* out_costs /* V or NULL */);
int32_t mnb_obstacle_reset(mnb_ctx* ctx);

/* lvr2::calcNormalClearance (clearance_layer.cpp:161): the free space above every vertex = distance along its normal
 * to the first face not incident to it, +inf if there is none; the input of the clearance cost mapping of
 * mnb_compute_layers.  vertex_normals: 3V floats or NULL = the normals mnb_set_mesh computed. */
int32_t mnb_normal_clearance(mnb_ctx* ctx, const float* vertex_normals, float* out_clearance /* V */);

/* ---- InflationLayer repulsive vector field -------------------------------------------------------------------------
 * vector_map_ as InflationLayer::waveFrontUpdate accumulates it (inflation_layer.cpp:277-308) for the LAST mnb_inflate /
 * mnb_inflation_update on this context; zero = no entry.  Derived from that wave's final labels, which live in the
 * workspace the planners share: call it before the next planner call on the context (MNB_E_STATE otherwise).  The field
 * and distances_ stay resident on the device.  out_vectors (3V) may be NULL. */
int32_t mnb_inflation_vector_map(mnb_ctx* ctx, float* out_vectors);
/* InflationLayer::vectorAt(vertices, barycentric_coords) (inflation_layer.cpp:493-521) of the resident field for n samples:
 * faces_q[n] face ids, bary[3n] -> out[3n]. */
int32_t mnb_inflation_vector_at(mnb_ctx* ctx, uint32_t n, const uint32_t* faces_q, const float* bary, float* out);
/* MeshMap::meshAhead adds every layer's vectorAt to the planner's direction (mesh_map.cpp:1097-1102): enable != 0 makes
 * mnb_cvp_backtrack add the resident inflation field (config_.repulsive_field, inflation_layer.h:247). */
int32_t mnb_set_repulsive_field(mnb_ctx* ctx, int32_t enable);

/* ---- cancel (CVPMeshPlanner::cancel / DijkstraMeshPlanner::cancel) ------- */
int32_t mnb_cancel(mnb_ctx* ctx);

/* ---- introspection for tests / bench ------------------------------------ */
typedef struct mnb_stats {
  uint64_t rounds;          /* band rounds of the last wavefront call */
  uint64_t recomputes;      /* vertex recomputations (>= settled vertices) */
  uint64_t settled;         /* vertices with a finite final label */
  uint64_t kernel_launches; /* kernels launched by the last call */
  float kernel_ms;          /* CUDA-event time of the wavefront kernel(s) of the last call */
  uint64_t skipped;         /* candidate-rounds that kept their label without a recompute (clean-candidate skip) */
  uint64_t deep_labels;     /* mnb_cvp: labels whose pop time has more than 3 nested cascade levels (informational: the order is exact at any depth; their level stacks live in the per-wavefront level pool) */
  uint64_t pool_words;      /* words of the level pool used by the last wavefront call (max over concurrent wavefronts) */
} mnb_stats;
int32_t mnb_get_stats(mnb_ctx* ctx, mnb_stats* out);
/* tuning knobs: band width delta (metres) and CTAs per wavefront cluster (1,2,4,8,16) */
int32_t mnb_set_tuning(mnb_ctx* ctx, float band_delta, int32_t cluster_size, int32_t threads_per_cta);

/* ---- multi-GPU: one host process, N devices (SURVEY.md 8e; north star: "batched multi-goal queries shard one goal per
 * GPU ... with NCCL over NVLink only to gather the resulting potential arrays") ----------------------------------------
 * A group owns one mnb_ctx per device (mnb_group_ctx: use it for everything that is per device -- layers, single plans,
 * tuning) and the NCCL communicators of the gather.  NCCL is bound at run time (libnccl.so.2); a group of one device
 * never touches it.  Reference counterpart: none -- the reference plans one query per MBF action on one CPU thread
 * (mbf_mesh_nav/src/mesh_planner_execution.cpp:55-66); this is the batched form of CVPMeshPlanner::waveFrontPropagation
 * (cvp_mesh_planner.cpp:651-886) behind mnb_cvp_batch, sharded. */
typedef struct mnb_group mnb_group;
int32_t mnb_group_create(int32_t n_devices, const int32_t* devices /* CUDA ordinals */, mnb_group** out_group);
void mnb_group_destroy(mnb_group* group);
int32_t mnb_group_size(mnb_group* group);
mnb_ctx* mnb_group_ctx(mnb_group* group, int32_t rank);
const char* mnb_group_last_error(mnb_group* group);
/* replicate the map / the per-plan costs on every device (HOST pointers, as mnb_set_mesh / mnb_set_costs) */
int32_t mnb_group_set_mesh(mnb_group* group, uint32_t V, uint32_t F, const float* pos, const uint32_t* faces,
                           const uint32_t* edges, uint32_t E);
int32_t mnb_group_set_costs(mnb_group* group, const float* vertex_costs, const float* edge_weights, const uint8_t* invalid);
/* MeshMap::layerChanged (mnb_update_vertex_costs) on every replica of the group, all devices concurrently; HOST arrays */
int32_t mnb_group_update_vertex_costs(mnb_group* group, uint32_t n_changed, const uint32_t* changed, const float* costs,
                                      int32_t costs_indexed_by_vertex, float default_value, double edge_cost_factor);
/* n full-field plans, goal k on rank k mod N, all devices concurrently; with gather != 0 one in-place ncclAllGather leaves
 * every field on every device.  Result on each device: float[N][pad][V], pad = ceil(n / N), the field of goal k is row
 * mnb_group_row(group, k); the buffers belong to the group and stay valid until its next sharded call.  seed arrays: HOST.
 * Returns the MBF code / MNB_E_* of the first rank that failed. */
int32_t mnb_cvp_batch_sharded(mnb_group* group, uint32_t n, const uint32_t* seed_faces, const float* seed_pos /* 3n */,
                              double cost_limit, int32_t gather);
uint32_t mnb_group_row(mnb_group* group, uint32_t goal);
float* mnb_group_fields(mnb_group* group, int32_t rank /* device pointer on that rank's device */);
int32_t mnb_group_read_fields(mnb_group* group, int32_t rank, uint32_t first_goal, uint32_t count, float* out_host /* count*V */);
/* n full-field Dijkstra plans (mnb_dijkstra_batch), sharded and gathered as mnb_cvp_batch_sharded: the distances go to the
 * same buffers in the same layout (mnb_group_row / mnb_group_fields / mnb_group_read_fields).  With want_pred != 0 the
 * predecessors go to a second group-owned buffer, uint32[N][pad][V] in the same layout, gathered together with the
 * distances in one NCCL group call.  seed array: HOST. */
int32_t mnb_dijkstra_batch_sharded(mnb_group* group, uint32_t n, const uint32_t* seed_vertices, double cost_limit,
                                   int32_t want_pred, int32_t gather);
uint32_t* mnb_group_preds(mnb_group* group, int32_t rank /* device pointer on that rank's device */);
/* MNB_E_STATE unless the last sharded call was mnb_dijkstra_batch_sharded with want_pred */
int32_t mnb_group_read_preds(mnb_group* group, int32_t rank, uint32_t first_goal, uint32_t count, uint32_t* out_host /* count*V */);

#ifdef __cplusplus
}
#endif
#endif /* MESHNAV_B200_H */
