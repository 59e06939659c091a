"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module.  The product package
(mesh_navigation_b200) never does.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "oracle.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"])
    return _SO


_lib = None


def use_native_build() -> str:
    """CPU-baseline legs of bench.py only: rebuild the oracle ON THIS HOST with `-O3 -march=native -DNDEBUG` (BASELINE.md
    section 2) into a temporary directory (the source tree may be read-only), removed at exit, and route every later call
    there.  The default liboracle.so is generic x86-64 because it may be built on another host than the one that runs it;
    -ffp-contract=off is kept, so results do not change.
    Returns the flag string actually in effect (the generic build if the native one cannot be compiled)."""
    global _SO, _lib
    out_dir = tempfile.mkdtemp(prefix="oracle_native_")
    atexit.register(shutil.rmtree, out_dir, ignore_errors=True)
    so = os.path.join(out_dir, "liboracle_native.so")
    flags = ["-O3", "-march=native", "-DNDEBUG", "-ffp-contract=off", "-fPIC", "-std=c++17"]
    try:
        subprocess.check_call(["g++"] + flags + ["-shared", "-o", so, os.path.join(_HERE, "oracle.cpp")],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=300)
        C.CDLL(so)                     # (an illegal-instruction build would have failed to compile, not to load; cheap check)
        _SO, _lib = so, None
        return "g++ " + " ".join(flags[:4])
    except Exception:
        return "g++ -O3 -DNDEBUG -ffp-contract=off (generic x86-64; native build failed)"


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        vp, u32, i64, dbl, f32 = C.c_void_p, C.c_uint32, C.c_int64, C.c_double, C.c_float
        L.orc_mesh_create.restype = vp
        L.orc_mesh_create.argtypes = [u32, u32, vp, vp, vp, u32]
        L.orc_mesh_destroy.argtypes = [vp]
        L.orc_mesh_num_edges.restype = u32
        L.orc_mesh_num_edges.argtypes = [vp]
        L.orc_mesh_get_edges.argtypes = [vp, vp]
        L.orc_edge_distances.argtypes = [vp, vp]
        L.orc_edge_weights.argtypes = [vp, vp, vp, dbl, vp]
        L.orc_dijkstra.restype = u32
        L.orc_dijkstra.argtypes = [vp, vp, vp, vp, u32, i64, dbl, dbl, C.c_int, vp, vp, vp]
        L.orc_cvp.restype = u32
        L.orc_cvp.argtypes = [vp, vp, vp, vp, u32, vp, i64, dbl, dbl, C.c_int, vp, vp, vp, vp, vp]
        L.orc_cvp_wavefront_update.restype = C.c_int
        L.orc_cvp_wavefront_update.argtypes = [vp, vp, u32, u32, u32, u32, vp, vp, vp, vp]
        L.orc_inflation_wavefront_update.restype = C.c_int
        L.orc_inflation_wavefront_update.argtypes = [vp, vp, vp, f32, vp, u32, u32, u32, u32]
        L.orc_fading.restype = f32
        L.orc_fading.argtypes = [dbl, dbl, dbl, dbl, dbl, f32]
        L.orc_sethian_update.restype = f32
        L.orc_sethian_update.argtypes = [f32] * 6
        L.orc_locate.argtypes = [vp, C.c_uint32, vp, vp, vp, vp]
        L.orc_cvp_backtrack.restype = C.c_int32
        L.orc_cvp_backtrack.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint32, C.c_double, C.c_uint32, vp, vp, vp]
        L.orc_dijkstra_vector_map.argtypes = [vp, vp, vp]
        L.orc_cvp_vector_map.argtypes = [vp, vp, vp, vp, vp, vp]
        L.orc_normals.argtypes = [vp, vp, vp]
        L.orc_layers.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.orc_inflation.argtypes = [vp, vp, vp, vp, u32, dbl, dbl, dbl, dbl, dbl, C.c_int, vp, vp, vp, vp]
        L.orc_layer_changed.argtypes = [vp, f32, vp, u32, vp]
        L.orc_update_edge_weights.argtypes = [vp, vp, vp, dbl, vp, u32, vp]
        L.orc_max_combination_update.argtypes = [u32, vp, vp, vp, vp, u32, vp, vp]
        L.orc_cast_rays.argtypes = [vp, u32, vp, vp, u32, vp, vp, vp, vp]
        L.orc_obstacle_update.argtypes = [vp, u32, vp, vp, vp, dbl, dbl, vp, vp]
        L.orc_normal_clearance.argtypes = [vp, vp, vp]
        L.orc_inflation_update_set.restype = u32
        L.orc_inflation_update_set.argtypes = [u32, vp, vp, vp]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class OracleMesh:
    def __init__(self, pos: np.ndarray, faces: np.ndarray, edges: np.ndarray | None = None):
        self.pos = np.ascontiguousarray(pos, dtype=np.float32).reshape(-1, 3)
        self.faces = np.ascontiguousarray(faces, dtype=np.uint32).reshape(-1, 3)
        self.V = self.pos.shape[0]
        self.F = self.faces.shape[0]
        e = None if edges is None else np.ascontiguousarray(edges, dtype=np.uint32).reshape(-1, 2)
        self._h = lib().orc_mesh_create(self.V, self.F, _p(self.pos), _p(self.faces), _p(e),
                                        0 if e is None else e.shape[0])
        self.E = lib().orc_mesh_num_edges(self._h)
        self.edges = np.empty((self.E, 2), dtype=np.uint32)
        lib().orc_mesh_get_edges(self._h, _p(self.edges))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_mesh_destroy(self._h)
            self._h = None

    def edge_distances(self) -> np.ndarray:
        out = np.empty(self.E, dtype=np.float32)
        lib().orc_edge_distances(self._h, _p(out))
        return out

    def edge_weights(self, vertex_costs, edge_distances, edge_cost_factor: float) -> np.ndarray:
        vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
        ed = np.ascontiguousarray(edge_distances, dtype=np.float32)
        out = np.empty(self.E, dtype=np.float32)
        lib().orc_edge_weights(self._h, _p(vc), _p(ed), float(edge_cost_factor), _p(out))
        return out

    def dijkstra(self, edge_weights, vertex_costs, seed_vertex: int, robot_vertex: int = -1,
                 invalid=None, cost_limit: float = 1.0, goal_dist_offset: float = 0.3, canonical_ties: bool = True):
        ew = np.ascontiguousarray(edge_weights, dtype=np.float32)
        vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        dist = np.empty(self.V, dtype=np.float32)
        pred = np.empty(self.V, dtype=np.uint32)
        stats = np.zeros(8, dtype=np.float64)
        rc = lib().orc_dijkstra(self._h, _p(ew), _p(vc), _p(inv), int(seed_vertex), int(robot_vertex),
                                float(cost_limit), float(goal_dist_offset), int(canonical_ties), _p(dist), _p(pred), _p(stats))
        return dict(outcome=rc, dist=dist, pred=pred, fixed=int(stats[0]), expanded=int(stats[1]),
                    seconds=float(stats[2]))

    def cvp(self, edge_weights, vertex_costs, seed_face: int, seed_pos, robot_face: int = -1,
            invalid=None, cost_limit: float = 1.0, goal_dist_offset: float = 0.3, canonical_ties: bool = True):
        ew = np.ascontiguousarray(edge_weights, dtype=np.float32)
        vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        sp = np.ascontiguousarray(seed_pos, dtype=np.float32)
        dist = np.empty(self.V, dtype=np.float32)
        pred = np.empty(self.V, dtype=np.uint32)
        direction = np.empty(self.V, dtype=np.float32)
        cut = np.empty(self.V, dtype=np.int32)
        stats = np.zeros(8, dtype=np.float64)
        rc = lib().orc_cvp(self._h, _p(ew), _p(vc), _p(inv), int(seed_face), _p(sp), int(robot_face),
                           float(cost_limit), float(goal_dist_offset), int(canonical_ties), _p(dist), _p(pred), _p(direction),
                           _p(cut), _p(stats))
        return dict(outcome=rc, dist=dist, pred=pred, direction=direction, cutting_face=cut,
                    fixed=int(stats[0]), expanded=int(stats[1]), seconds=float(stats[2]),
                    updates=int(stats[3]), accepted=int(stats[4]), backsteps=int(stats[5]),
                    max_backstep=float(stats[6]))

    def cvp_wavefront_update(self, edge_weights, face, v1, v2, v3, dist, pred, direction, cut) -> bool:
        ew = np.ascontiguousarray(edge_weights, dtype=np.float32)
        return bool(lib().orc_cvp_wavefront_update(self._h, _p(ew), face, v1, v2, v3, _p(dist), _p(pred),
                                                   _p(direction), _p(cut)))

    def inflation_wavefront_update(self, dist, vectors, max_distance, edge_weights, face, v1, v2, v3) -> bool:
        ew = np.ascontiguousarray(edge_weights, dtype=np.float32)
        return bool(lib().orc_inflation_wavefront_update(self._h, _p(dist), _p(vectors), float(max_distance),
                                                         _p(ew), face, v1, v2, v3))

    def inflation(self, edge_distances, lethals, invalid=None, inscribed_radius=0.25, inflation_radius=0.4,
                  lethal_value=1.0, inscribed_value=0.99, cost_scaling_factor=1.0, with_vectors=False,
                  canonical_ties: bool = True):
        ed = np.ascontiguousarray(edge_distances, dtype=np.float32)
        le = np.unique(np.ascontiguousarray(lethals, dtype=np.uint32))  # std::set order
        inv = None if invalid is None else np.ascontiguousarray(invalid, dtype=np.uint8)
        dist = np.empty(self.V, dtype=np.float32)
        cost = np.empty(self.V, dtype=np.float32)
        vec = np.zeros((self.V, 3), dtype=np.float32) if with_vectors else None
        stats = np.zeros(8, dtype=np.float64)
        lib().orc_inflation(self._h, _p(ed), _p(inv), _p(le), le.size, float(inscribed_radius),
                            float(inflation_radius), float(lethal_value), float(inscribed_value),
                            float(cost_scaling_factor), int(canonical_ties), _p(dist), _p(cost), _p(vec), _p(stats))
        return dict(dist=dist, cost=cost, vectors=vec, pops=int(stats[0]), seconds=float(stats[1]),
                    updates=int(stats[2]))


def _layer_changed(layer_costs, default_value, changed, vertex_costs):
    """MeshMap::layerChanged (mesh_map.cpp:478-487): vertex_costs updated in place for the changed vertices."""
    lc = np.ascontiguousarray(layer_costs, dtype=np.float32)
    ch = np.unique(np.ascontiguousarray(changed, dtype=np.uint32))
    assert vertex_costs.dtype == np.float32 and vertex_costs.flags.c_contiguous
    lib().orc_layer_changed(_p(lc), C.c_float(default_value), _p(ch), ch.size, _p(vertex_costs))
    return vertex_costs


def _update_edge_weights(self, vertex_costs, edge_distances, edge_cost_factor, changed, edge_weights):
    """MeshMap::updateEdgeWeights (mesh_map.cpp:563-618): edge_weights updated in place."""
    vc = np.ascontiguousarray(vertex_costs, dtype=np.float32)
    ed = np.ascontiguousarray(edge_distances, dtype=np.float32)
    ch = np.unique(np.ascontiguousarray(changed, dtype=np.uint32))
    assert edge_weights.dtype == np.float32 and edge_weights.flags.c_contiguous
    lib().orc_update_edge_weights(self._h, _p(vc), _p(ed), C.c_double(edge_cost_factor), _p(ch), ch.size, _p(edge_weights))
    return edge_weights


def max_combination_update(layer_costs, defaults, layer_lethals, changed, costs, lethals=None):
    """MaxCombinationLayer::onInputChanged (combination_layer.cpp:87-147): costs / lethals updated in place."""
    L = len(layer_costs)
    lcs = [np.ascontiguousarray(a, dtype=np.float32) for a in layer_costs]
    lls = [None if a is None else np.ascontiguousarray(a, dtype=np.uint8) for a in layer_lethals]
    cp = (C.c_void_p * L)(*[a.ctypes.data for a in lcs])
    lp = (C.c_void_p * L)(*[None if a is None else a.ctypes.data for a in lls])
    df = np.ascontiguousarray(defaults, dtype=np.float32)
    ch = np.unique(np.ascontiguousarray(changed, dtype=np.uint32))
    lib().orc_max_combination_update(L, cp, _p(df), lp, _p(ch), ch.size, _p(costs), _p(lethals))
    return costs, lethals


def avg_combination_update(layer_costs, defaults, weights, layer_lethals, changed, costs, lethals=None):
    """AvgCombinationLayer::onInputChanged / computeLayer (combination_layer.cpp:185-302): costs / lethals updated in place."""
    L = len(layer_costs)
    lcs = [np.ascontiguousarray(a, dtype=np.float32) for a in layer_costs]
    lls = [None if a is None else np.ascontiguousarray(a, dtype=np.uint8) for a in layer_lethals]
    cp = (C.c_void_p * L)(*[a.ctypes.data for a in lcs])
    lp = (C.c_void_p * L)(*[None if a is None else a.ctypes.data for a in lls])
    df = np.ascontiguousarray(defaults, dtype=np.float32); wt = np.ascontiguousarray(weights, dtype=np.float32)
    ch = np.unique(np.ascontiguousarray(changed, dtype=np.uint32))
    f = lib().orc_avg_combination_update
    f.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    f(L, cp, _p(df), _p(wt), lp, _p(ch), ch.size, _p(costs), _p(lethals))
    return costs, lethals


def inflation_update_set(new_costs, old_costs=None):
    """InflationLayer::onInputChanged (inflation_layer.cpp:154-164): keys(new) U keys(old), ascending."""
    nc = np.ascontiguousarray(new_costs, dtype=np.float32)
    oc = None if old_costs is None else np.ascontiguousarray(old_costs, dtype=np.float32)
    out = np.empty(nc.size, dtype=np.uint32)
    lib().orc_inflation_update_set.restype = C.c_uint32
    n = lib().orc_inflation_update_set(nc.size, _p(nc), _p(oc), _p(out))
    return out[:n].copy()


layer_changed = _layer_changed


class LayerParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "height_diff_threshold", "height_diff_radius", "roughness_threshold", "roughness_radius", "steepness_threshold",
        "ridge_threshold", "ridge_radius", "clearance_robot_height", "clearance_height_inflation", "border_threshold",
        "border_cost")]

    @staticmethod
    def defaults():
        return LayerParams(0.185, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3, 0.5, 0.3, 0.5, 1.0)


LAYER_NAMES = ["height_diff", "roughness", "steepness", "ridge", "clearance", "border"]


def _layers(self, params=None, clearance=None):
    P = params or LayerParams.defaults()
    fn = np.empty((self.F, 3), np.float32); vn = np.empty((self.V, 3), np.float32)
    lib().orc_normals(self._h, _p(fn), _p(vn))
    outs = [np.empty(self.V, np.float32) for _ in range(6)]
    comb = np.empty(self.V, np.float32); mask = np.empty(self.V, np.uint8)
    cl = None if clearance is None else np.ascontiguousarray(clearance, dtype=np.float32)
    lib().orc_layers(self._h, C.byref(P), _p(vn), _p(cl), *[_p(o) for o in outs], _p(comb), _p(mask))
    r = dict(zip(LAYER_NAMES, outs))
    r.update(combined=comb, lethal_mask=mask, vertex_normals=vn, face_normals=fn)
    return r


OracleMesh.layers = _layers
OracleMesh.update_edge_weights = _update_edge_weights


def _dijkstra_vector_map(self, pred):
    out = np.empty((self.V, 3), np.float32)
    lib().orc_dijkstra_vector_map(self._h, _p(np.ascontiguousarray(pred, dtype=np.uint32)), _p(out))
    return out


def _cvp_vector_map(self, vertex_normals, pred, direction, cutting_face):
    out = np.empty((self.V, 3), np.float32)
    lib().orc_cvp_vector_map(self._h, _p(np.ascontiguousarray(vertex_normals, dtype=np.float32)),
                             _p(np.ascontiguousarray(pred, dtype=np.uint32)), _p(np.ascontiguousarray(direction, dtype=np.float32)),
                             _p(np.ascontiguousarray(cutting_face, dtype=np.int32)), _p(out))
    return out


def _cvp_backtrack(self, vector_map, start, start_face, goal, goal_face, step_width=0.4, max_points=100000, repulsive=None):
    """cvp:920-951: walk from `goal` (robot) down the field to `start` (wave seed); returns (outcome, positions, faces).
    repulsive: optional dict(dist, vectors, inscribed_radius, inflation_radius, lethal_value, inscribed_value) -- the
    InflationLayer field meshAhead adds (mesh_map.cpp:1097-1102, inflation_layer.cpp:493-521)"""
    vm = np.ascontiguousarray(vector_map, dtype=np.float32)
    st = np.ascontiguousarray(start, dtype=np.float32); go = np.ascontiguousarray(goal, dtype=np.float32)
    pp = np.empty((max_points, 3), np.float32); pf = np.empty(max_points, np.uint32); n = C.c_uint32(0)
    if repulsive is not None:
        rd = np.ascontiguousarray(repulsive["dist"], dtype=np.float32); rv = np.ascontiguousarray(repulsive["vectors"], dtype=np.float32)
        f = lib().orc_cvp_backtrack_repulsive
        f.restype = C.c_int32
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_double, C.c_uint32, C.c_void_p,
                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double]
        rc = f(self._h, _p(vm), _p(st), int(start_face), _p(go), int(goal_face), float(step_width), int(max_points), _p(pp),
               _p(pf), C.byref(n), _p(rd), _p(rv), float(repulsive.get("inscribed_radius", 0.25)),
               float(repulsive.get("inflation_radius", 0.4)), float(repulsive.get("lethal_value", 1.0)),
               float(repulsive.get("inscribed_value", 0.99)))
        k = min(n.value, max_points)
        return rc, pp[:k].copy(), pf[:k].copy()
    rc = lib().orc_cvp_backtrack(self._h, _p(vm), _p(st), int(start_face), _p(go), int(goal_face), float(step_width),
                                 int(max_points), _p(pp), _p(pf), C.byref(n))
    k = min(n.value, max_points)
    return rc, pp[:k].copy(), pf[:k].copy()


def _locate(self, points):
    """getNearestVertexHandle + searchContainingFace (mesh_map.cpp:1120-1174) -> (vertex, face or -1, bary)"""
    pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    n = pts.shape[0]
    nv = np.empty(n, np.uint32); fc = np.empty(n, np.int32); ba = np.empty((n, 3), np.float32)
    lib().orc_locate(self._h, n, _p(pts), _p(nv), _p(fc), _p(ba))
    return nv, fc, ba


def _inflation_vector_at(self, faces_q, bary, dist, vectors, inscribed_radius=0.25, inflation_radius=0.4, lethal_value=1.0,
                         inscribed_value=0.99):
    """InflationLayer::vectorAt(vertices, barycentric_coords) (inflation_layer.cpp:493-521) for n samples"""
    fq = np.ascontiguousarray(faces_q, dtype=np.uint32); ba = np.ascontiguousarray(bary, dtype=np.float32).reshape(-1, 3)
    rd = np.ascontiguousarray(dist, dtype=np.float32); rv = np.ascontiguousarray(vectors, dtype=np.float32)
    out = np.empty((fq.size, 3), np.float32)
    f = lib().orc_inflation_vector_at
    f.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double,
                  C.c_double, C.c_void_p]
    f(self._h, fq.size, _p(fq), _p(ba), _p(rd), _p(rv), float(inscribed_radius), float(inflation_radius), float(lethal_value),
      float(inscribed_value), _p(out))
    return out


OracleMesh.inflation_vector_at = _inflation_vector_at
OracleMesh.locate = _locate
OracleMesh.cvp_backtrack = _cvp_backtrack
OracleMesh.dijkstra_vector_map = _dijkstra_vector_map
OracleMesh.cvp_vector_map = _cvp_vector_map


def fading(distance, inscribed_radius=0.25, inflation_radius=0.4, lethal_value=1.0, inscribed_value=0.99,
           cost_scaling_factor=1.0) -> float:
    return float(lib().orc_fading(inscribed_radius, inflation_radius, lethal_value, inscribed_value,
                                  cost_scaling_factor, float(distance)))


def _cast_rays(self, origins, dirs):
    """orc_cast_rays: brute-force nearest hit of every ray (dirs [3] = one direction for all rays)"""
    o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(dirs, dtype=np.float32)
    stride = 0 if d.size == 3 and o.shape[0] != 1 else 3
    n = o.shape[0]
    hit = np.empty(n, np.uint8); dist = np.empty(n, np.float32); face = np.empty(n, np.uint32); point = np.empty((n, 3), np.float32)
    lib().orc_cast_rays(self._h, n, _p(o), _p(d), stride, _p(hit), _p(dist), _p(face), _p(point))
    return dict(hit=hit, dist=dist, face=face, point=point)


def _obstacle_update(self, points, tf, axis, max_obstacle_dist, robot_height, lethal_mask):
    """orc_obstacle_update: lethal_mask (V bytes) is rolled over in place; returns (new lethal ids, changed ids), ascending"""
    pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    T = np.ascontiguousarray(tf, dtype=np.float32).reshape(12)
    ax = np.ascontiguousarray(axis, dtype=np.float32).reshape(3)
    changed = np.zeros(self.V, np.uint8)
    lib().orc_obstacle_update(self._h, pts.shape[0], _p(pts), _p(T), _p(ax), float(max_obstacle_dist), float(robot_height),
                              _p(lethal_mask), _p(changed))
    return np.nonzero(lethal_mask)[0].astype(np.uint32), np.nonzero(changed)[0].astype(np.uint32)


def _normal_clearance(self, vertex_normals):
    vn = np.ascontiguousarray(vertex_normals, dtype=np.float32).reshape(-1, 3)
    out = np.empty(self.V, np.float32)
    lib().orc_normal_clearance(self._h, _p(vn), _p(out))
    return out


OracleMesh.cast_rays = _cast_rays
OracleMesh.obstacle_update = _obstacle_update
OracleMesh.normal_clearance = _normal_clearance
