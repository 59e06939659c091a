"""GPU parity tests of the ray caster (SURVEY.md 8 row f3 remainder): mnb_cast_rays, ObstacleLayer::processPointCloud
(obstacle_layer.cpp:215-296) and lvr2::calcNormalClearance (clearance_layer.cpp:161) -- through the C ABI, bit for bit
against the oracle's brute-force loop over all faces (oracle.cpp "Ray casting against the map").  The BVH of the product
may only change the cost of a query, never its result.  (Also replayed on the CPU interpreter of the kernels.)"""
import numpy as np
import pytest

from tests.util import delaunay_mesh, mesh_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from mesh_navigation_b200 import api as A
    return A


def two_storey(n=40, m=18, gap=1.2, tilt=0.15):
    """terrain with a tilted roof patch above its middle: rays from below hit the roof, rays from above hit roof or ground"""
    pos, faces = mesh_case(n, True)
    rpos, rfaces = mesh_case(m, False, seed=5)
    rpos = rpos.copy()
    off = (n - m) * 0.05
    rpos[:, 0] += off; rpos[:, 1] += off
    rpos[:, 2] = float(pos[:, 2].max()) + gap + tilt * (rpos[:, 0] - off)
    return np.vstack([pos, rpos]).astype(np.float32), np.vstack([faces, rfaces + pos.shape[0]]).astype(np.uint32)


def same_hits(got, ref):
    assert (got["hit"] == ref["hit"]).all()
    assert (got["face"] == ref["face"]).all()
    assert (got["dist"].view(np.uint32) == ref["dist"].view(np.uint32)).all()
    assert (got["point"].view(np.uint32) == ref["point"].view(np.uint32)).all()


def test_cast_rays_bit_identical_to_brute_force(api, oracle_mod):
    pos, faces = two_storey()
    om = oracle_mod.OracleMesh(pos, faces); mm = api.MeshMap(pos, faces)
    rng = np.random.default_rng(3)
    lo, hi = pos.min(0) - 0.5, pos.max(0) + 0.5
    n = 1500
    o = (lo + rng.random((n, 3)) * (hi - lo)).astype(np.float32)
    d = rng.normal(size=(n, 3)); d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    # axis-parallel rays (zero components take the slab test's flat branch), rays that start exactly above a vertex and hit
    # it (every incident face reports the same t: the smallest face id must win), rays along edges, a zero direction
    d[:60] = np.array([0, 0, -1], np.float32); d[60:90] = np.array([0, 0, 1], np.float32)
    d[90:110] = np.array([1, 0, 0], np.float32); d[110:130] = np.array([0, -1, 0], np.float32)
    vs = rng.integers(0, pos.shape[0], 40)
    o[:40] = pos[vs] + np.array([0, 0, 0.75], np.float32)
    e0 = faces[rng.integers(0, faces.shape[0], 20)]
    o[130:150] = pos[e0[:, 0]]; dd = pos[e0[:, 1]] - pos[e0[:, 0]]
    d[130:150] = (dd / np.linalg.norm(dd, axis=1, keepdims=True)).astype(np.float32)
    d[150] = 0.0
    got = mm.castRays(o, d); ref = om.cast_rays(o, d)
    same_hits(got, ref)
    assert 200 < int(ref["hit"].sum()) < n                      # hits and misses both occur
    assert (ref["hit"][:40] == 1).all()
    # one shared direction (obstacle_layer.cpp:229)
    down = np.array([0, 0, -1], np.float32)
    same_hits(mm.castRays(o, down), om.cast_rays(o, down))
    # no rays
    assert mm.castRays(np.zeros((0, 3), np.float32), down)["hit"].size == 0
    mm.close()


def test_cast_rays_irregular_mesh_and_coarse_morton_cells(api, oracle_mod):
    """a Delaunay mesh plus one far-away triangle: the scene box becomes huge, thousands of faces share a Morton cell and
    the radix tree has to split them by position -- the results must still be those of the loop over all faces"""
    pos, faces = delaunay_mesh(900, seed=5)
    pos = pos.copy(); pos[:, 2] = 0.3 * np.sin(pos[:, 0]) * np.cos(1.3 * pos[:, 1])
    far = np.array([[4.0e6, 4.0e6, 10.0], [4.0e6 + 1, 4.0e6, 10.0], [4.0e6, 4.0e6 + 1, 10.0]], np.float32)
    pos2 = np.vstack([pos, far]).astype(np.float32)
    faces2 = np.vstack([faces, np.array([[pos.shape[0], pos.shape[0] + 1, pos.shape[0] + 2]], np.uint32)]).astype(np.uint32)
    for P, Fc in ((pos.astype(np.float32), faces), (pos2, faces2)):
        om = oracle_mod.OracleMesh(P, Fc); mm = api.MeshMap(P, Fc)
        rng = np.random.default_rng(8)
        n = 800
        o = np.empty((n, 3), np.float32)
        o[:, :2] = rng.random((n, 2)) * 6.0; o[:, 2] = rng.random(n) * 2.0 - 0.5
        d = rng.normal(size=(n, 3)); d[:, 2] -= 1.0
        d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
        same_hits(mm.castRays(o, d), om.cast_rays(o, d))
        mm.close()


@pytest.mark.parametrize("nfaces", [1, 2])
def test_cast_rays_tiny_meshes(api, oracle_mod, nfaces):
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.2]], np.float32)
    faces = np.array([[0, 1, 2], [1, 3, 2]], np.uint32)[:nfaces]
    pos = pos[:3 + (nfaces - 1)]
    om = oracle_mod.OracleMesh(pos, faces); mm = api.MeshMap(pos, faces)
    o = np.array([[0.2, 0.2, 1], [0.8, 0.8, 1], [2, 2, 1], [0.5, 0.5, -1], [0.25, 0.25, 0.0]], np.float32)
    d = np.array([[0, 0, -1], [0, 0, -1], [0, 0, -1], [0, 0, 1], [0, 0, -1]], np.float32)
    got = mm.castRays(o, d)
    same_hits(got, om.cast_rays(o, d))
    assert got["hit"][0] == 1 and got["hit"][2] == 0 and got["hit"][4] == 1 and got["dist"][4] == 0.0     # a point on the surface hits at t = 0
    mm.close()


def test_obstacle_layer_point_clouds(api, oracle_mod):
    """three consecutive clouds through ObstacleLayer::processPointCloud: range filter, message -> map transform, ray
    along the rotated down axis, height filter, lethal set and changed set (symmetric difference with the previous set)"""
    pos, faces = two_storey()
    om = oracle_mod.OracleMesh(pos, faces); mm = api.MeshMap(pos, faces)
    layer = api.ObstacleLayer(mm, robot_height=0.8, max_obstacle_dist=2.5)
    mask = np.zeros(om.V, np.uint8)
    rng = np.random.default_rng(21)
    centre = pos[:, :2].mean(0)
    seen_changed = 0
    for step in range(4):
        n = [4000, 2500, 0, 1500][step]                          # the empty cloud clears the set: everything changes back
        pts = (rng.normal(size=(n, 3)) * np.array([1.2, 1.2, 0.6])).astype(np.float32)
        if n:
            pts[::97] = np.nan                                   # invalid returns are dropped by the range filter
            pts[5::50] *= 4.0                                    # beyond max_obstacle_dist
        ang = 0.3 * step
        R = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]], np.float32)
        t = np.array([centre[0] + 0.2 * step, centre[1] - 0.1 * step, float(pos[:, 2].mean()) + 1.0], np.float32)
        T = np.hstack([R, t[:, None]]).astype(np.float32)
        tilt = np.array([0.05 * step, -0.03 * step, -1.0], np.float32); axis = (tilt / np.linalg.norm(tilt)).astype(np.float32)
        ref_le, ref_ch = om.obstacle_update(pts, T, axis, 2.5, 0.8, mask)
        got = layer.processPointCloud(pts, T, axis, want_costs=True)
        assert np.array_equal(got["lethals"], ref_le), step
        assert np.array_equal(got["changed"], ref_ch), step
        assert np.isinf(got["costs"][ref_le]).all() and np.isnan(np.delete(got["costs"], ref_le)).all()
        seen_changed += ref_ch.size
        if step == 0:
            assert ref_le.size > 50
        if step == 2:
            assert ref_le.size == 0 and ref_ch.size > 0
    assert seen_changed > 100
    mm.close()


def test_normal_clearance_and_clearance_layer(api, oracle_mod):
    """calcNormalClearance under the roof: finite clearances below it, +inf in the open; the clearance cost mapping of the
    fused layer kernel then marks the low headroom lethal (clearance_layer.cpp:67-99)"""
    pos, faces = two_storey(gap=0.45, tilt=0.02)
    om = oracle_mod.OracleMesh(pos, faces); mm = api.MeshMap(pos, faces)
    vn = mm.vertexNormals()
    ref = om.normal_clearance(vn)
    got = mm.normalClearance(vn)
    assert (got.view(np.uint32) == ref.view(np.uint32)).all()
    assert (mm.normalClearance().view(np.uint32) == ref.view(np.uint32)).all()     # NULL = the map's own normals
    fin = np.isfinite(ref)
    assert 100 < int(fin.sum()) < om.V - 100
    # degenerate normals: no ray
    vn2 = vn.copy(); vn2[::7] = 0.0; vn2[3::11] = np.nan
    ref2 = om.normal_clearance(vn2); got2 = mm.normalClearance(vn2)
    assert (got2.view(np.uint32) == ref2.view(np.uint32)).all() and np.isinf(ref2[::7]).all()
    from mesh_navigation_b200 import _lib
    h = float(np.median(ref[fin]))                               # half of the vertices under the roof are too low
    P = oracle_mod.LayerParams.defaults(); P.clearance_robot_height = h
    G = _lib.LayerParams.defaults(); G.clearance_robot_height = h
    L = mm.computeLayers(G, got); R = om.layers(P, ref)
    assert (L["clearance"].view(np.uint32) == R["clearance"].view(np.uint32)).all()
    assert (L["lethal_mask"] == R["lethal_mask"]).all()
    assert int((L["clearance"] == 1.0).sum()) > 20
    mm.close()


def test_obstacle_update_with_device_resident_arrays(api, oracle_mod):
    """MNB_PTR_DEVICE: the cloud, the lethal list and the changed list stay on the device (what a device-resident layer stack
    feeds into mnb_inflation_update); only the two counts come back.  Same sets as the host-pointer call and as the oracle."""
    import ctypes as C
    pos, faces = two_storey()
    om = oracle_mod.OracleMesh(pos, faces); mm = api.MeshMap(pos, faces)
    rng = np.random.default_rng(4)
    pts = (rng.normal(size=(3000, 3)) * np.array([1.0, 1.0, 0.5])).astype(np.float32)
    centre = pos[:, :2].mean(0)
    T = np.float32([[1, 0, 0, centre[0]], [0, 1, 0, centre[1]], [0, 0, 1, float(pos[:, 2].mean()) + 1.0]])
    ax = np.float32([0, 0, -1])
    mask = np.zeros(om.V, np.uint8)
    ref_le, ref_ch = om.obstacle_update(pts, T, ax, 3.0, 0.9, mask)
    # the loaded library decides, not torch: the CPU interpreter of the kernels (tests/emu, the only build that exports
    # mnb_emu_switch) dereferences "device" pointers on the host, also on a machine that has a GPU
    on_gpu = not hasattr(mm.L, "mnb_emu_switch")
    if on_gpu:      # a real device: torch owns the buffers
        import torch
        d_pts = torch.from_numpy(pts).cuda(); d_le = torch.empty(om.V, dtype=torch.int32, device="cuda"); d_ch = torch.empty(om.V, dtype=torch.int32, device="cuda")
        ptr = lambda t: C.c_void_p(t.data_ptr()); back = lambda t, n: t[:n].cpu().numpy().view(np.uint32)
    else:           # the CPU interpreter of the kernels: "device" memory is host memory
        d_pts = pts.copy(); d_le = np.empty(om.V, np.uint32); d_ch = np.empty(om.V, np.uint32)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p); back = lambda a, n: a[:n].copy()
    cfg = api._lib.ObstacleParams(); cfg.max_obstacle_dist = 3.0; cfg.robot_height = 0.9
    cfg.tf[:] = [float(x) for x in T.reshape(-1)]; cfg.down_axis[:] = [0.0, 0.0, -1.0]
    assert mm.L.mnb_obstacle_reset(mm._ctx) == 0
    nl, nc = C.c_uint32(0), C.c_uint32(0)
    mm.use_device_pointers(True)
    try:
        rc = mm.L.mnb_obstacle_update(mm._ctx, pts.shape[0], ptr(d_pts), C.byref(cfg), ptr(d_le), C.byref(nl), ptr(d_ch), C.byref(nc), None)
    finally:
        mm.use_device_pointers(False)
    assert rc == 0
    assert np.array_equal(back(d_le, nl.value), ref_le) and np.array_equal(back(d_ch, nc.value), ref_ch) and ref_le.size > 50
    mm.close()
