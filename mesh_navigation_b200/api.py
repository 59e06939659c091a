"""Thin Python driver over the C ABI (test / bench orchestration only).

Mirrors the names of the reference's hot-path entry points:
  MeshMap.computeEdgeWeights      mesh_map/src/mesh_map.cpp:517-561
  DijkstraMeshPlanner.dijkstra    dijkstra_mesh_planner/src/dijkstra_mesh_planner.cpp:217-398
  CVPMeshPlanner.waveFrontPropagation  cvp_mesh_planner/src/cvp_mesh_planner.cpp:651-886
  InflationLayer.waveCostInflation     mesh_layers/src/inflation_layer.cpp:341-491
All compute happens in libmeshnav_b200.so on the GPU; nothing here falls back to
numpy or to the oracle.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


class MeshNavError(RuntimeError):
    pass


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


class MeshMap:
    """Device-resident flattened mesh + the per-plan inputs the planners read
    (vertex_costs, edge_weights, invalid) -- the slice of mesh_map::MeshMap the hot path touches."""

    def __init__(self, pos: np.ndarray, faces: np.ndarray, edges: np.ndarray | None = None, device: int = 0):
        self.L = _lib.load()
        self._ctx = C.c_void_p()
        rc = self.L.mnb_create(device, C.byref(self._ctx))
        if rc != 0:
            raise MeshNavError(f"mnb_create failed ({rc}): no usable sm_100 CUDA device; there is no CPU fallback")
        self.pos = np.ascontiguousarray(pos, dtype=np.float32).reshape(-1, 3)
        self.faces = np.ascontiguousarray(faces, dtype=np.uint32).reshape(-1, 3)
        e = None if edges is None else np.ascontiguousarray(edges, dtype=np.uint32).reshape(-1, 2)
        self._check(self.L.mnb_set_mesh(self._ctx, self.pos.shape[0], self.faces.shape[0], _p(self.pos), _p(self.faces),
                                        _p(e), 0 if e is None else e.shape[0]))
        self.V = self.L.mnb_num_vertices(self._ctx)
        self.F = self.L.mnb_num_faces(self._ctx)
        self.E = self.L.mnb_num_edges(self._ctx)
        self.device_pointers = False

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self.L.mnb_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise MeshNavError(f"meshnav_b200 error {rc}: {self.L.mnb_last_error(self._ctx).decode()}")
        return rc

    # -- setup ------------------------------------------------------------
    def set_tuning(self, band_delta: float = 0.0, cluster_size: int = 0, threads: int = 0):
        self._check(self.L.mnb_set_tuning(self._ctx, band_delta, cluster_size, threads))

    def use_device_pointers(self, on: bool):
        self._check(self.L.mnb_set_pointer_mode(self._ctx, 1 if on else 0))
        self.device_pointers = on

    def stream(self) -> int:
        return int(self.L.mnb_stream(self._ctx) or 0)

    def edges(self) -> np.ndarray:
        out = np.empty((self.E, 2), dtype=np.uint32)
        self._check(self.L.mnb_get_edges(self._ctx, _p(out)))
        return out

    def edgeDistances(self) -> np.ndarray:
        assert not self.device_pointers
        out = np.empty(self.E, dtype=np.float32)
        self._check(self.L.mnb_get_edge_distances(self._ctx, _p(out)))
        return out

    def computeEdgeWeights(self, vertex_costs, edge_cost_factor: float = 0.0, want_output: bool = True):
        vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
        out = np.empty(self.E, dtype=np.float32) if want_output else None
        self._check(self.L.mnb_compute_edge_weights(self._ctx, _p(vc), float(edge_cost_factor), _p(out)))
        return out

    def setCosts(self, vertex_costs, edge_weights, invalid=None):
        if self.device_pointers:
            self._check(self.L.mnb_set_costs(self._ctx, _p(vertex_costs), _p(edge_weights), _p(invalid)))
            return
        vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
        ew = np.ascontiguousarray(edge_weights, dtype=np.float32)
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        assert vc.size == self.V and ew.size == self.E
        self._check(self.L.mnb_set_costs(self._ctx, _p(vc), _p(ew), _p(inv)))

    # -- incremental updates (SURVEY.md 3.4) ---------------------------------
    def layerChanged(self, changed, costs, edge_cost_factor: float, by_vertex: bool = False, default_value: float = 0.0):
        """MeshMap::layerChanged + updateEdgeWeights (mesh_map.cpp:455-492, 563-618) for the changed vertices only.
        costs: one value per changed vertex, or (by_vertex) the default layer's V-sized map with NaN = no entry"""
        if self.device_pointers:
            ch, n = changed
            return self._check(self.L.mnb_update_vertex_costs(self._ctx, int(n), _p(ch), _p(costs), int(by_vertex),
                                                              float(default_value), float(edge_cost_factor)))
        ch = np.ascontiguousarray(changed, dtype=np.uint32)
        co = np.ascontiguousarray(costs, dtype=np.float32)
        assert co.size == (self.V if by_vertex else ch.size)
        return self._check(self.L.mnb_update_vertex_costs(self._ctx, ch.size, _p(ch), _p(co), int(by_vertex),
                                                          float(default_value), float(edge_cost_factor)))

    def costs(self):
        """(vertex_costs, edge_weights) as installed on the device"""
        vc = np.empty(self.V, dtype=np.float32); ew = np.empty(self.E, dtype=np.float32)
        self._check(self.L.mnb_get_costs(self._ctx, _p(vc), _p(ew)))
        return vc, ew

    def maxCombinationUpdate(self, layer_costs, defaults, layer_lethals, changed, io_costs, io_lethal=None, weights=None):
        """MaxCombinationLayer::onInputChanged (combination_layer.cpp:87-147), or with `weights`
        AvgCombinationLayer::onInputChanged (:250-302): io_costs / io_lethal updated in place"""
        n = len(layer_costs)
        lcs = [np.ascontiguousarray(a, dtype=np.float32) for a in layer_costs]
        lls = [None if a is None else np.ascontiguousarray(a, dtype=np.uint8) for a in (layer_lethals or [None] * n)]
        cp = (C.c_void_p * n)(*[a.ctypes.data for a in lcs])
        lp = (C.c_void_p * n)(*[None if a is None else a.ctypes.data for a in lls])
        df = np.ascontiguousarray(defaults, dtype=np.float32)
        ch = np.ascontiguousarray(changed, dtype=np.uint32)
        assert io_costs.dtype == np.float32 and io_costs.flags.c_contiguous and io_costs.size == self.V
        if weights is not None:
            wt = np.ascontiguousarray(weights, dtype=np.float32)
            self._check(self.L.mnb_avg_combination_update(self._ctx, n, cp, _p(df), _p(wt), lp, ch.size, _p(ch), _p(io_costs), _p(io_lethal)))
        else:
            self._check(self.L.mnb_max_combination_update(self._ctx, n, cp, _p(df), lp, ch.size, _p(ch), _p(io_costs), _p(io_lethal)))
        return io_costs, io_lethal

    def avgCombinationUpdate(self, layer_costs, defaults, weights, layer_lethals, changed, io_costs, io_lethal=None):
        return self.maxCombinationUpdate(layer_costs, defaults, layer_lethals, changed, io_costs, io_lethal, weights=weights)

    def vertexNormals(self) -> np.ndarray:
        out = np.empty((self.V, 3), dtype=np.float32)
        self._check(self.L.mnb_get_vertex_normals(self._ctx, _p(out)))
        return out

    def computeLayers(self, params=None, clearance=None) -> dict:
        """the six geometric layers + MaxCombinationLayer + lethal masks in one fused kernel"""
        P = params or _lib.LayerParams.defaults()
        cl = None if clearance is None else np.ascontiguousarray(clearance, dtype=np.float32)
        costs = np.empty((6, self.V), dtype=np.float32)
        comb = np.empty(self.V, dtype=np.float32)
        mask = np.empty(self.V, dtype=np.uint8)
        self._check(self.L.mnb_compute_layers(self._ctx, C.byref(P), _p(cl), _p(costs), _p(comb), _p(mask)))
        r = {n: costs[i] for i, n in enumerate(_lib.LAYER_NAMES)}
        r.update(combined=comb, lethal_mask=mask, **self.stats())
        return r

    def castRays(self, origins, dirs):
        """the map's shared raycaster (MeshMap::raycaster()->castRays, mesh_map.h:318 / obstacle_layer.cpp:239): one unit
        direction per ray ([n,3]) or one for all ([3]); returns hit flags, distances, face ids, hit points"""
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, dtype=np.float32)
        stride = 0 if d.size == 3 and o.shape[0] != 1 else 3
        if stride == 3 and d.size != o.size:
            raise ValueError("dirs must be [3] or [n,3]")
        n = o.shape[0]
        hit = np.empty(n, np.uint8); dist = np.empty(n, np.float32); face = np.empty(n, np.uint32); point = np.empty((n, 3), np.float32)
        self._check(self.L.mnb_cast_rays(self._ctx, n, _p(o), _p(d), stride, _p(hit), _p(dist), _p(face), _p(point)))
        return dict(hit=hit, dist=dist, face=face, point=point, **self.stats())

    def normalClearance(self, vertex_normals=None) -> np.ndarray:
        """lvr2::calcNormalClearance (clearance_layer.cpp:161): free space above every vertex along its normal"""
        vn = None if vertex_normals is None else np.ascontiguousarray(vertex_normals, dtype=np.float32)
        out = np.empty(self.V, dtype=np.float32)
        self._check(self.L.mnb_normal_clearance(self._ctx, _p(vn), _p(out)))
        return out

    def locate(self, points):
        """getNearestVertexHandle + searchContainingFace (mesh_map.cpp:1110-1174) for a batch of points ->
        (nearest vertex u32[n], containing face i32[n] (-1 none), barycentric coords f32[n,3])"""
        pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        n = pts.shape[0]
        nv = np.empty(n, np.uint32); fc = np.empty(n, np.int32); ba = np.empty((n, 3), np.float32)
        self._check(self.L.mnb_locate(self._ctx, n, _p(pts), _p(nv), _p(fc), _p(ba)))
        return nv, fc, ba

    def getNearestVertexHandle(self, p) -> int:
        return int(self.locate(p)[0][0])

    def getContainingFace(self, p, max_dist: float = 0.4) -> int:
        """-1 = no containing face; max_dist is accepted and (like the reference, mesh_map.cpp:1120-1159) not consulted"""
        return int(self.locate(p)[1][0])

    def vectorMap(self, pred, direction=None, cutting_face=None) -> np.ndarray:
        """computeVectorMap of the planners (dijkstra:189-209 with direction=None, cvp:204-239 otherwise)"""
        pr = np.ascontiguousarray(pred, dtype=np.uint32)
        di = None if direction is None else np.ascontiguousarray(direction, dtype=np.float32)
        cu = None if cutting_face is None else np.ascontiguousarray(cutting_face, dtype=np.int32)
        out = np.empty((self.V, 3), dtype=np.float32)
        self._check(self.L.mnb_vector_map(self._ctx, _p(pr), _p(di), _p(cu), _p(out)))
        return out

    def stats(self) -> dict:
        s = _lib.Stats()
        self._check(self.L.mnb_get_stats(self._ctx, C.byref(s)))
        return dict(rounds=s.rounds, recomputes=s.recomputes, settled=s.settled, kernel_launches=s.kernel_launches,
                    kernel_ms=s.kernel_ms, skipped=s.skipped, deep_labels=s.deep_labels)

    def cancel(self):
        self._check(self.L.mnb_cancel(self._ctx))

    # -- raw device-pointer entry points (bench "value" leg) ---------------
    def dijkstra_dev(self, seed_vertex, robot_vertex, cost_limit, goal_dist_offset, d_dist: int, d_pred: int) -> int:
        return self._check(self.L.mnb_dijkstra(self._ctx, int(seed_vertex), int(robot_vertex), float(cost_limit),
                                               float(goal_dist_offset), _p(d_dist), _p(d_pred)))

    def cvp_dev(self, seed_face, seed_pos, robot_face, cost_limit, goal_dist_offset, d_dist: int, d_pred: int = 0,
                d_dir: int = 0, d_cut: int = 0) -> int:
        sp = np.ascontiguousarray(seed_pos, dtype=np.float32)
        return self._check(self.L.mnb_cvp(self._ctx, int(seed_face), _p(sp), int(robot_face), float(cost_limit),
                                          float(goal_dist_offset), _p(d_dist) if d_dist else None,
                                          _p(d_pred) if d_pred else None, _p(d_dir) if d_dir else None,
                                          _p(d_cut) if d_cut else None))

    def cvp_batch_dev(self, seed_faces, seed_pos, cost_limit, d_out: int) -> int:
        sf = np.ascontiguousarray(seed_faces, dtype=np.uint32)
        sp = np.ascontiguousarray(seed_pos, dtype=np.float32).reshape(-1, 3)
        return self._check(self.L.mnb_cvp_batch(self._ctx, sf.size, _p(sf), _p(sp), float(cost_limit), _p(d_out)))

    def dijkstra_batch_dev(self, seed_vertices, cost_limit, d_dist: int, d_pred: int = 0) -> int:
        """mnb_dijkstra_batch into device rows [n][V] (needs use_device_pointers(True)); d_pred = 0: no predecessors"""
        sv = np.ascontiguousarray(seed_vertices, dtype=np.uint32).ravel()
        return self._check(self.L.mnb_dijkstra_batch(self._ctx, sv.size, _p(sv), float(cost_limit), _p(d_dist),
                                                     _p(d_pred) if d_pred else None))


class DijkstraMeshPlanner:
    """dijkstra_mesh_planner::DijkstraMeshPlanner -- wavefront part (dijkstra():217-398)."""

    def __init__(self, mesh_map: MeshMap, cost_limit: float = 1.0, goal_dist_offset: float = 0.3):
        self.map = mesh_map
        self.cost_limit = cost_limit                # dijkstra_mesh_planner.h:178-187
        self.goal_dist_offset = goal_dist_offset

    def dijkstra(self, seed_vertex: int, robot_vertex: int = -1):
        m = self.map
        dist = np.empty(m.V, dtype=np.float32)
        pred = np.empty(m.V, dtype=np.uint32)
        rc = m._check(m.L.mnb_dijkstra(m._ctx, int(seed_vertex), int(robot_vertex), float(self.cost_limit),
                                       float(self.goal_dist_offset), _p(dist), _p(pred)))
        return dict(outcome=rc, dist=dist, pred=pred, **m.stats())

    def dijkstraBatch(self, seed_vertices, want_pred: bool = True):
        """full-field dijkstra() for many goals in one call (mnb_dijkstra_batch): row k of dist / pred is what
        dijkstra(seed_vertices[k]) returns; the vector field of goal k is computeVectorMap(pred[k])"""
        m = self.map
        sv = np.ascontiguousarray(seed_vertices, dtype=np.uint32).ravel()
        dist = np.empty((sv.size, m.V), dtype=np.float32)
        pred = np.empty((sv.size, m.V), dtype=np.uint32) if want_pred else None
        rc = m._check(m.L.mnb_dijkstra_batch(m._ctx, sv.size, _p(sv), float(self.cost_limit), _p(dist), _p(pred)))
        return dict(outcome=rc, dist=dist, pred=pred, **m.stats())

    def computeVectorMap(self, pred):
        return self.map.vectorMap(pred)


class CVPMeshPlanner:
    """cvp_mesh_planner::CVPMeshPlanner -- wavefront part (waveFrontPropagation():651-886)."""

    def __init__(self, mesh_map: MeshMap, cost_limit: float = 1.0, goal_dist_offset: float = 0.3):
        self.map = mesh_map
        self.cost_limit = cost_limit                # cvp_mesh_planner.h:201-212
        self.goal_dist_offset = goal_dist_offset

    def waveFrontPropagation(self, seed_face: int, seed_pos, robot_face: int = -1, out=None):
        """out: optional dict of preallocated host arrays (dist f32, pred u32, direction f32, cutting_face i32), e.g.
        views of pinned memory, that receive the results"""
        m = self.map
        sp = np.ascontiguousarray(seed_pos, dtype=np.float32)
        dist = out["dist"] if out else np.empty(m.V, dtype=np.float32)
        pred = out["pred"] if out else np.empty(m.V, dtype=np.uint32)
        direction = out["direction"] if out else np.empty(m.V, dtype=np.float32)
        cut = out["cutting_face"] if out else np.empty(m.V, dtype=np.int32)
        rc = m._check(m.L.mnb_cvp(m._ctx, int(seed_face), _p(sp), int(robot_face), float(self.cost_limit),
                                  float(self.goal_dist_offset), _p(dist), _p(pred), _p(direction), _p(cut)))
        return dict(outcome=rc, dist=dist, pred=pred, direction=direction, cutting_face=cut, **m.stats())

    def computeVectorMap(self, pred, direction, cutting_face):
        return self.map.vectorMap(pred, direction, cutting_face)

    def backtrack(self, robot_pos, robot_face: int, step_width: float = 0.4, max_points: int = 1 << 16):
        """vector-field back-tracking of the last waveFrontPropagation (cvp:920-951 / MeshMap::meshAhead), on the GPU;
        returns the poses in plan order (robot first, wave seed last)"""
        m = self.map
        rp = np.ascontiguousarray(robot_pos, dtype=np.float32)
        pos = np.empty((max_points, 3), dtype=np.float32); face = np.empty(max_points, dtype=np.uint32)
        n = C.c_uint32(0)
        rc = m._check(m.L.mnb_cvp_backtrack(m._ctx, _p(rp), int(robot_face), float(step_width), int(max_points), _p(pos),
                                            _p(face), C.byref(n)))
        return dict(outcome=rc, positions=pos[:n.value].copy(), faces=face[:n.value].copy(), **m.stats())

    def makePlan(self, start_pos, start_face: int, goal_pos, goal_face: int, step_width: float = 0.4):
        """CVPMeshPlanner::makePlan (cvp:62-140): the wave is seeded at the GOAL and runs until the robot (start) face is
        fixed; only the path comes back to the host.  cost = sum of the segment lengths (cvp:104-120)"""
        m = self.map
        sp = np.ascontiguousarray(goal_pos, dtype=np.float32)
        rc = m._check(m.L.mnb_cvp(m._ctx, int(goal_face), _p(sp), int(start_face), float(self.cost_limit),
                                  float(self.goal_dist_offset), None, None, None, None))
        st = m.stats()
        if rc != 0:
            return dict(outcome=rc, positions=np.empty((0, 3), np.float32), faces=np.empty(0, np.uint32), cost=0.0, **st)
        bt = self.backtrack(start_pos, start_face, step_width)
        p = bt["positions"]
        cost = float(np.linalg.norm(np.diff(p, axis=0), axis=1).sum()) if len(p) > 1 else 0.0
        bt.update(cost=cost, wavefront_ms=st["kernel_ms"])
        return bt

    def waveFrontPropagationBatch(self, seed_faces, seed_pos):
        m = self.map
        sf = np.ascontiguousarray(seed_faces, dtype=np.uint32)
        sp = np.ascontiguousarray(seed_pos, dtype=np.float32).reshape(-1, 3)
        out = np.empty((sf.size, m.V), dtype=np.float32)
        rc = m._check(m.L.mnb_cvp_batch(m._ctx, sf.size, _p(sf), _p(sp), float(self.cost_limit), _p(out)))
        return dict(outcome=rc, dist=out, **m.stats())


class InflationLayer:
    """mesh_layers::InflationLayer -- waveCostInflation (inflation_layer.cpp:341-491)."""

    def __init__(self, mesh_map: MeshMap, inscribed_radius=0.25, inflation_radius=0.4, lethal_value=1.0,
                 inscribed_value=0.99, cost_scaling_factor=1.0):
        self.map = mesh_map
        self.config = _lib.InflationParams(inscribed_radius, inflation_radius, lethal_value, inscribed_value,
                                           cost_scaling_factor)   # inflation_layer.h:240-248

    def waveCostInflation(self, lethals, invalid=None):
        m = self.map
        le = np.ascontiguousarray(lethals, dtype=np.uint32)
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        dist = np.empty(m.V, dtype=np.float32)
        cost = np.empty(m.V, dtype=np.float32)
        m._check(m.L.mnb_inflate(m._ctx, _p(le), le.size, _p(inv), C.byref(self.config), _p(dist), _p(cost)))
        return dict(dist=dist, cost=cost, **m.stats())

    def vectorMap(self) -> np.ndarray:
        """vector_map_ of the last wave (inflation_layer.cpp:277-308), [V,3], zero = no entry; call before the next plan"""
        m = self.map
        out = np.empty((m.V, 3), dtype=np.float32)
        m._check(m.L.mnb_inflation_vector_map(m._ctx, _p(out)))
        return out

    def vectorAt(self, faces_q, bary) -> np.ndarray:
        """InflationLayer::vectorAt(vertices, barycentric_coords) (inflation_layer.cpp:493-521) for n samples"""
        m = self.map
        fq = np.ascontiguousarray(faces_q, dtype=np.uint32); ba = np.ascontiguousarray(bary, dtype=np.float32).reshape(-1, 3)
        out = np.empty((fq.size, 3), dtype=np.float32)
        m._check(m.L.mnb_inflation_vector_at(m._ctx, fq.size, _p(fq), _p(ba), _p(out)))
        return out

    def setRepulsiveField(self, on: bool):
        """config_.repulsive_field: meshAhead (the planners' back-tracking) adds this layer's vectorAt"""
        self.map._check(self.map.L.mnb_set_repulsive_field(self.map._ctx, int(bool(on))))

    def onInputChanged(self, lethals, invalid=None):
        """InflationLayer::onInputChanged (inflation_layer.cpp:97-179): full re-inflation + the update set
        (vertices with a riskiness entry now or after the previous inflation on this map, ascending)"""
        m = self.map
        le = np.ascontiguousarray(lethals, dtype=np.uint32)
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        dist = np.empty(m.V, dtype=np.float32)
        cost = np.empty(m.V, dtype=np.float32)
        changed = np.empty(m.V, dtype=np.uint32)
        n = C.c_uint32(0)
        m._check(m.L.mnb_inflation_update(m._ctx, _p(le), le.size, _p(inv), C.byref(self.config), _p(dist), _p(cost),
                                          _p(changed), C.byref(n)))
        return dict(dist=dist, cost=cost, changed=changed[:n.value].copy(), **m.stats())


class ObstacleLayer:
    """mesh_layers::ObstacleLayer (obstacle_layer.cpp): the lethal set of the latest point cloud"""

    def __init__(self, mesh_map: MeshMap, robot_height: float = 1.0, max_obstacle_dist: float = 10.0, down_axis=(0.0, 0.0, -1.0)):
        self.map = mesh_map
        self.config = _lib.ObstacleParams()
        self.config.robot_height = robot_height; self.config.max_obstacle_dist = max_obstacle_dist
        ax = np.asarray(down_axis, dtype=np.float32)
        ax = ax / np.float32(np.linalg.norm(ax))                      # config_.down_axis is normalised (obstacle_layer.cpp:110)
        self.down_axis = ax
        self.map._check(self.map.L.mnb_obstacle_reset(self.map._ctx))

    def processPointCloud(self, points, tf=None, down_axis_map=None, want_costs: bool = False):
        """ObstacleLayer::processPointCloud (obstacle_layer.cpp:133-296): `points` in the message frame, `tf` the 3x4 [R|t]
        into the map frame (identity if None), `down_axis_map` the down axis rotated into the map frame (the configured
        axis if None).  Returns the new lethal set, the changed set (ascending) and optionally the cost map."""
        m = self.map
        pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        T = np.hstack([np.eye(3, dtype=np.float32), np.zeros((3, 1), np.float32)]) if tf is None else np.asarray(tf, dtype=np.float32).reshape(3, 4)
        ax = self.down_axis if down_axis_map is None else np.asarray(down_axis_map, dtype=np.float32)
        self.config.tf[:] = [float(x) for x in T.reshape(-1)]
        self.config.down_axis[:] = [float(x) for x in ax]
        lethals = np.empty(m.V, np.uint32); changed = np.empty(m.V, np.uint32)
        costs = np.empty(m.V, np.float32) if want_costs else None
        nl, nc = C.c_uint32(0), C.c_uint32(0)
        m._check(m.L.mnb_obstacle_update(m._ctx, pts.shape[0], _p(pts), C.byref(self.config), _p(lethals), C.byref(nl), _p(changed),
                                         C.byref(nc), _p(costs)))
        out = dict(lethals=lethals[:nl.value].copy(), changed=changed[:nc.value].copy(), **m.stats())
        if want_costs:
            out["costs"] = costs
        return out
