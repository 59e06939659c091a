"""ctypes binding of libmeshnav_b200.so (include/meshnav_b200.h).

There is no fallback: if the shared library is missing or no sm_100 device is
usable, importing works but every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmeshnav_b200.so")

MNB_OK = 0
MNB_PTR_HOST = 0
MNB_PTR_DEVICE = 1
OUTCOME = {0: "SUCCESS", 51: "CANCELED", 52: "INVALID_START", 53: "INVALID_GOAL", 54: "NO_PATH_FOUND"}


class InflationParams(C.Structure):
    _fields_ = [("inscribed_radius", C.c_double), ("inflation_radius", C.c_double), ("lethal_value", C.c_double),
                ("inscribed_value", C.c_double), ("cost_scaling_factor", C.c_double)]


class ObstacleParams(C.Structure):
    """ObstacleLayer config (mesh_layers/include/mesh_layers/obstacle_layer.h) + the two transforms of one message"""
    _fields_ = [("max_obstacle_dist", C.c_double), ("robot_height", C.c_double), ("tf", C.c_float * 12), ("down_axis", C.c_float * 3)]


class LayerParams(C.Structure):
    """config structs at the end of mesh_layers/include/mesh_layers/*_layer.h (doubles)"""
    _fields_ = [(n, C.c_double) for n in (
        "height_diff_threshold", "height_diff_radius", "roughness_threshold", "roughness_radius", "steepness_threshold",
        "ridge_threshold", "ridge_radius", "clearance_robot_height", "clearance_height_inflation", "border_threshold",
        "border_cost")]

    @staticmethod
    def defaults():
        return LayerParams(0.185, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3, 0.5, 0.3, 0.5, 1.0)


LAYER_NAMES = ["height_diff", "roughness", "steepness", "ridge", "clearance", "border"]


class Stats(C.Structure):
    _fields_ = [("rounds", C.c_uint64), ("recomputes", C.c_uint64), ("settled", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("kernel_ms", C.c_float), ("skipped", C.c_uint64), ("deep_labels", C.c_uint64), ("pool_words", C.c_uint64)]


# every symbol include/meshnav_b200.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "mnb_create", "mnb_destroy", "mnb_last_error", "mnb_set_pointer_mode", "mnb_stream", "mnb_set_mesh",
    "mnb_num_vertices", "mnb_num_faces", "mnb_num_edges", "mnb_get_edges", "mnb_get_edge_distances",
    "mnb_compute_edge_weights", "mnb_set_costs", "mnb_dijkstra", "mnb_dijkstra_batch", "mnb_cvp", "mnb_cvp_batch", "mnb_inflate",
    "mnb_cancel", "mnb_get_stats", "mnb_set_tuning", "mnb_compute_layers", "mnb_get_vertex_normals", "mnb_vector_map", "mnb_cvp_backtrack", "mnb_locate",
    "mnb_update_vertex_costs", "mnb_get_costs", "mnb_max_combination_update", "mnb_avg_combination_update", "mnb_inflation_update",
    "mnb_inflation_vector_map", "mnb_inflation_vector_at", "mnb_set_repulsive_field",
    "mnb_cast_rays", "mnb_obstacle_update", "mnb_obstacle_reset", "mnb_normal_clearance",
    "mnb_group_create", "mnb_group_destroy", "mnb_group_size", "mnb_group_ctx", "mnb_group_last_error", "mnb_group_set_mesh",
    "mnb_group_set_costs", "mnb_group_update_vertex_costs", "mnb_cvp_batch_sharded", "mnb_group_row", "mnb_group_fields", "mnb_group_read_fields",
    "mnb_dijkstra_batch_sharded", "mnb_group_preds", "mnb_group_read_preds",
]

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                           "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, u32, i64, dbl, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_int64, C.c_double, C.c_float
    L.mnb_create.restype = i32; L.mnb_create.argtypes = [i32, C.POINTER(vp)]
    L.mnb_destroy.restype = None; L.mnb_destroy.argtypes = [vp]
    L.mnb_last_error.restype = C.c_char_p; L.mnb_last_error.argtypes = [vp]
    L.mnb_set_pointer_mode.restype = i32; L.mnb_set_pointer_mode.argtypes = [vp, i32]
    L.mnb_stream.restype = vp; L.mnb_stream.argtypes = [vp]
    L.mnb_set_mesh.restype = i32; L.mnb_set_mesh.argtypes = [vp, u32, u32, vp, vp, vp, u32]
    for f in ("mnb_num_vertices", "mnb_num_faces", "mnb_num_edges"):
        getattr(L, f).restype = u32; getattr(L, f).argtypes = [vp]
    L.mnb_get_edges.restype = i32; L.mnb_get_edges.argtypes = [vp, vp]
    L.mnb_get_edge_distances.restype = i32; L.mnb_get_edge_distances.argtypes = [vp, vp]
    L.mnb_compute_edge_weights.restype = i32; L.mnb_compute_edge_weights.argtypes = [vp, vp, dbl, vp]
    L.mnb_set_costs.restype = i32; L.mnb_set_costs.argtypes = [vp, vp, vp, vp]
    L.mnb_dijkstra.restype = i32; L.mnb_dijkstra.argtypes = [vp, u32, i64, dbl, dbl, vp, vp]
    L.mnb_dijkstra_batch.restype = i32; L.mnb_dijkstra_batch.argtypes = [vp, u32, vp, dbl, vp, vp]
    L.mnb_cvp.restype = i32; L.mnb_cvp.argtypes = [vp, u32, vp, i64, dbl, dbl, vp, vp, vp, vp]
    L.mnb_cvp_batch.restype = i32; L.mnb_cvp_batch.argtypes = [vp, u32, vp, vp, dbl, vp]
    L.mnb_inflate.restype = i32; L.mnb_inflate.argtypes = [vp, vp, u32, vp, C.POINTER(InflationParams), vp, vp]
    L.mnb_compute_layers.restype = i32; L.mnb_compute_layers.argtypes = [vp, C.POINTER(LayerParams), vp, vp, vp, vp]
    L.mnb_get_vertex_normals.restype = i32; L.mnb_get_vertex_normals.argtypes = [vp, vp]
    L.mnb_vector_map.restype = i32; L.mnb_vector_map.argtypes = [vp, vp, vp, vp, vp]
    L.mnb_locate.restype = i32; L.mnb_locate.argtypes = [vp, u32, vp, vp, vp, vp]
    L.mnb_cvp_backtrack.restype = i32
    L.mnb_cvp_backtrack.argtypes = [vp, vp, C.c_uint32, C.c_double, C.c_uint32, vp, vp, vp]
    L.mnb_update_vertex_costs.restype = i32; L.mnb_update_vertex_costs.argtypes = [vp, u32, vp, vp, i32, f32, dbl]
    L.mnb_get_costs.restype = i32; L.mnb_get_costs.argtypes = [vp, vp, vp]
    L.mnb_max_combination_update.restype = i32
    L.mnb_max_combination_update.argtypes = [vp, u32, vp, vp, vp, u32, vp, vp, vp]
    L.mnb_avg_combination_update.restype = i32
    L.mnb_avg_combination_update.argtypes = [vp, u32, vp, vp, vp, vp, u32, vp, vp, vp]
    L.mnb_inflation_update.restype = i32
    L.mnb_inflation_update.argtypes = [vp, vp, u32, vp, C.POINTER(InflationParams), vp, vp, vp, C.POINTER(C.c_uint32)]
    L.mnb_inflation_vector_map.restype = i32; L.mnb_inflation_vector_map.argtypes = [vp, vp]
    L.mnb_inflation_vector_at.restype = i32; L.mnb_inflation_vector_at.argtypes = [vp, u32, vp, vp, vp]
    L.mnb_set_repulsive_field.restype = i32; L.mnb_set_repulsive_field.argtypes = [vp, i32]
    L.mnb_cast_rays.restype = i32; L.mnb_cast_rays.argtypes = [vp, u32, vp, vp, u32, vp, vp, vp, vp]
    L.mnb_obstacle_update.restype = i32
    L.mnb_obstacle_update.argtypes = [vp, u32, vp, C.POINTER(ObstacleParams), vp, C.POINTER(C.c_uint32), vp, C.POINTER(C.c_uint32), vp]
    L.mnb_obstacle_reset.restype = i32; L.mnb_obstacle_reset.argtypes = [vp]
    L.mnb_normal_clearance.restype = i32; L.mnb_normal_clearance.argtypes = [vp, vp, vp]
    L.mnb_cancel.restype = i32; L.mnb_cancel.argtypes = [vp]
    L.mnb_get_stats.restype = i32; L.mnb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.mnb_set_tuning.restype = i32; L.mnb_set_tuning.argtypes = [vp, f32, i32, i32]
    _lib = L
    return L
