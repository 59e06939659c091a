"""Batched full-field Dijkstra (mnb_dijkstra_batch, DijkstraMeshPlanner.dijkstraBatch, mnb_dijkstra_batch_sharded): every
row of every batch must equal the oracle's DijkstraMeshPlanner::dijkstra of that goal -- distances bit for bit,
predecessors exactly -- and, where exact key ties exist, the single-plan mnb_dijkstra row by row."""
import ctypes as C

import numpy as np
import pytest

from mesh_navigation_b200 import synth
from tests.util import delaunay_mesh, mesh_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from mesh_navigation_b200 import api as A
    return A


def make(api, oracle_mod, pos, faces, costs=None, factor=0.0, invalid=None):
    om = oracle_mod.OracleMesh(pos, faces)
    mm = api.MeshMap(pos, faces)
    ed = om.edge_distances()
    vc = np.zeros(om.V, np.float32) if costs is None else costs.astype(np.float32)
    w = om.edge_weights(vc, ed, factor)
    mm.setCosts(vc, w, invalid)
    return om, mm, ed, vc, w


def check_rows(om, got, seeds, w, vc, invalid=None, cost_limit=1.0):
    assert got["outcome"] == 0
    assert got["dist"].shape == (len(seeds), om.V)
    for k, s in enumerate(seeds):
        ref = om.dijkstra(w, vc, int(s), invalid=invalid, cost_limit=cost_limit)
        assert (got["dist"][k].view(np.uint32) == ref["dist"].view(np.uint32)).all(), ("dist", k, int(s))
        if got["pred"] is not None:
            assert (got["pred"][k] == ref["pred"]).all(), ("pred", k, int(s))


@pytest.mark.parametrize("n,terrain,goals,cluster", [(40, False, 11, 0), (36, True, 9, 0), (30, True, 1, 0), (34, True, 6, 2), (32, False, 5, 4)])
def test_batch_matches_oracle_jittered(api, oracle_mod, n, terrain, goals, cluster):
    """cluster 0: CTAs per goal chosen from the goal count; 2 / 4: fixed by mnb_set_tuning"""
    pos, faces = mesh_case(n, terrain)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    mm.set_tuning(0.0, cluster, 0)
    seeds = np.random.default_rng(n).integers(0, om.V, goals).astype(np.uint32)
    got = api.DijkstraMeshPlanner(mm).dijkstraBatch(seeds)
    check_rows(om, got, seeds, w, vc)
    assert got["kernel_launches"] == 1 and got["rounds"] > 0 and got["recomputes"] > 0
    assert got["settled"] == goals * om.V                      # every vertex of a connected mesh is reached by every goal
    mm.close()


def test_batch_unjittered_ties_match_single_plans(api, oracle_mod):
    """exact key ties (regular grid): the argmin on the converged row must pick what the heap loop's pop order picks"""
    pos, faces = synth.grid_mesh(24, 24, jitter=0.0)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    seeds = np.array([0, 300, 575, 17, 288], np.uint32)
    P = api.DijkstraMeshPlanner(mm)
    got = P.dijkstraBatch(seeds)
    check_rows(om, got, seeds, w, vc)
    for k, s in enumerate(seeds):
        one = P.dijkstra(int(s))
        assert (got["dist"][k].view(np.uint32) == one["dist"].view(np.uint32)).all() and (got["pred"][k] == one["pred"]).all(), k
    mm.close()


def test_batch_high_degree_csr_path(api, oracle_mod):
    """a hub vertex of degree 24 (> the 8 ELL slots) relaxes and is relaxed through the CSR lists"""
    pos, faces = delaunay_mesh(500, with_hub=True)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    hub = om.V - 1
    seeds = np.array([hub, 0, 250, int(faces[0][1])], np.uint32)
    check_rows(om, api.DijkstraMeshPlanner(mm).dijkstraBatch(seeds), seeds, w, vc)
    mm.close()


def test_batch_costs_invalid_disconnected_inf_weights(api, oracle_mod):
    """cost wall above cost_limit (labelled, not expanded), invalid vertices and an invalid seed (expanded, as the reference
    does), a second component (unreached: +inf / self), +inf edge weights from +inf vertex costs"""
    pos1, faces1 = mesh_case(26, True)
    pos2 = pos1[:100] + np.array([20.0, 0, 0], np.float32)
    faces2 = faces1[(faces1 < 100).all(1)]
    pos = np.concatenate([pos1, pos2]); faces = np.concatenate([faces1, faces2 + len(pos1)]).astype(np.uint32)
    rng = np.random.default_rng(5)
    V = len(pos)
    vc = (rng.random(V) * 0.8).astype(np.float32)
    vc[(pos[:, 0] > 1.2) & (pos[:, 0] < 1.4) & (pos[:, 1] < 1.8)] = 1.5       # wall with a gap
    vc[rng.choice(V, 12, replace=False)] = np.inf
    invalid = (rng.random(V) < 0.02).astype(np.uint8)
    seeds = np.array([3, 400, len(pos1) + 10, 600], np.uint32)
    invalid[seeds[0]] = 1
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces, costs=vc, factor=1.0, invalid=invalid)
    assert np.isinf(w).any()
    got = api.DijkstraMeshPlanner(mm).dijkstraBatch(seeds)
    check_rows(om, got, seeds, w, vc, invalid=invalid)
    assert np.isinf(got["dist"][0][len(pos1):]).all() and (got["pred"][0][len(pos1):] == np.arange(len(pos1), V)).all()
    assert np.isinf(got["dist"][2][:len(pos1)]).all()
    mm.close()


def test_batch_queue_ragged_and_duplicate_seeds(api, oracle_mod):
    """more goals than resident CTA slots (148 SMs x 4): persistent groups take goals from the queue; duplicates allowed"""
    pos, faces = mesh_case(12, True)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    seeds = np.random.default_rng(9).integers(0, om.V, 1203).astype(np.uint32)
    seeds[7] = seeds[8] = seeds[1000]
    got = api.DijkstraMeshPlanner(mm).dijkstraBatch(seeds)
    refs = {int(s): om.dijkstra(w, vc, int(s)) for s in np.unique(seeds)}
    for k, s in enumerate(seeds):
        assert (got["dist"][k].view(np.uint32) == refs[int(s)]["dist"].view(np.uint32)).all(), k
        assert (got["pred"][k] == refs[int(s)]["pred"]).all(), k
    mm.close()


def test_batch_without_pred_and_device_pointers(api, oracle_mod):
    pos, faces = mesh_case(30, False)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    seeds = np.array([5, 450, 899], np.uint32)
    P = api.DijkstraMeshPlanner(mm)
    nopred = P.dijkstraBatch(seeds, want_pred=False)
    assert nopred["pred"] is None
    check_rows(om, nopred, seeds, w, vc)
    # device-pointer mode: the loaded library decides, not torch (the CPU interpreter of the kernels dereferences "device"
    # pointers on the host)
    on_gpu = not hasattr(mm.L, "mnb_emu_switch")
    if on_gpu:
        import torch
        d_dist = torch.empty((len(seeds), om.V), dtype=torch.float32, device="cuda")
        d_pred = torch.empty((len(seeds), om.V), dtype=torch.int32, device="cuda")
        ptr = lambda t: t.data_ptr(); back = lambda t: t.cpu().numpy()
    else:           # (host memory is shared with the interpreter's CTAs only when they run in the caller: no clusters)
        mm.set_tuning(0.0, 1, 0)
        d_dist = np.empty((len(seeds), om.V), np.float32); d_pred = np.empty((len(seeds), om.V), np.int32)
        ptr = lambda a: a.ctypes.data; back = lambda a: a.copy()
    mm.use_device_pointers(True)
    assert mm.dijkstra_batch_dev(seeds, 1.0, ptr(d_dist), ptr(d_pred)) == 0
    dev = dict(outcome=0, dist=back(d_dist), pred=back(d_pred).view(np.uint32))
    check_rows(om, dev, seeds, w, vc)
    assert mm.dijkstra_batch_dev(seeds[::-1], 1.0, ptr(d_dist), 0) == 0       # out_pred NULL: pred rows untouched
    assert (back(d_dist)[0].view(np.uint32) == dev["dist"][2].view(np.uint32)).all()
    assert (back(d_pred).view(np.uint32) == dev["pred"]).all()
    mm.use_device_pointers(False)
    mm.close()


def test_batch_after_vertex_cost_update(api, oracle_mod):
    """mnb_update_vertex_costs patches the weights in place; the batch rebuilds its adjacency tables and plans on them"""
    pos, faces = mesh_case(32, True)
    rng = np.random.default_rng(2)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces, costs=rng.random(len(pos)) * 0.5, factor=1.0)
    seeds = np.array([40, 700, 1000], np.uint32)
    P = api.DijkstraMeshPlanner(mm)
    check_rows(om, P.dijkstraBatch(seeds), seeds, w, vc)
    ch = rng.choice(om.V, om.V // 5, replace=False).astype(np.uint32)
    nv = (rng.random(ch.size) * 1.4).astype(np.float32)
    mm.layerChanged(ch, nv, 1.0)
    vc2 = vc.copy(); vc2[ch] = nv
    w2 = w.copy(); om.update_edge_weights(vc2, ed, 1.0, ch, w2)
    check_rows(om, P.dijkstraBatch(seeds), seeds, w2, vc2)
    mm.close()


def test_batch_leaves_the_last_cvp_result_alone(api, oracle_mod):
    """mnb_cvp -> mnb_dijkstra_batch -> mnb_cvp_backtrack returns the path of mnb_cvp -> mnb_cvp_backtrack"""
    pos, faces = mesh_case(40, True)
    om, mm, ed, vc, w = make(api, oracle_mod, pos, faces)
    cvp = api.CVPMeshPlanner(mm)
    sf, rf = 100, 2800
    sp, rp = pos[faces[sf]].mean(0), pos[faces[rf]].mean(0)
    assert cvp.waveFrontPropagation(sf, sp)["outcome"] == 0
    a = cvp.backtrack(rp, rf)
    assert cvp.waveFrontPropagation(sf, sp)["outcome"] == 0
    api.DijkstraMeshPlanner(mm).dijkstraBatch(np.arange(0, om.V, 97, dtype=np.uint32))
    b = cvp.backtrack(rp, rf)
    assert a["outcome"] == b["outcome"] == 0 and len(a["positions"]) > 2
    assert np.array_equal(a["positions"], b["positions"]) and np.array_equal(a["faces"], b["faces"])
    mm.close()


def test_batch_error_codes(api, oracle_mod):
    pos, faces = mesh_case(10, False)
    mm = api.MeshMap(pos, faces)
    L = mm.L
    one = np.zeros(1, np.uint32)
    dist = np.empty((1, mm.V), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.mnb_dijkstra_batch(mm._ctx, 1, p(one), 1.0, p(dist), None) == -3           # MNB_E_STATE: no costs yet
    mm.setCosts(np.zeros(mm.V, np.float32), mm.edgeDistances())
    assert L.mnb_dijkstra_batch(mm._ctx, 0, p(one), 1.0, p(dist), None) == -1           # MNB_E_ARG: n = 0
    assert L.mnb_dijkstra_batch(mm._ctx, 1, None, 1.0, p(dist), None) == -1
    assert L.mnb_dijkstra_batch(mm._ctx, 1, p(one), 1.0, None, None) == -1
    bad = np.array([0, mm.V], np.uint32)
    out = np.full((2, mm.V), 7.0, np.float32)
    assert L.mnb_dijkstra_batch(mm._ctx, 2, p(bad), 1.0, p(out), None) == 52           # MNB_INVALID_START, nothing written
    assert (out == 7.0).all()
    mm.close()


def test_sharded_dijkstra_batch_through_the_c_abi(oracle_mod):
    """mirrors test_gpu_group.py: goal k on rank k mod N, fields and predecessors gathered onto every rank"""
    import torch
    from mesh_navigation_b200 import _lib
    L = _lib.load()
    ndev = max(1, min(2, torch.cuda.device_count())) if not hasattr(L, "mnb_emu_switch") else 1
    pos, faces = mesh_case(40, True)
    om = oracle_mod.OracleMesh(pos, faces)
    ed = om.edge_distances(); vc = np.zeros(om.V, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for f in ("mnb_group_create", "mnb_group_set_mesh", "mnb_group_set_costs", "mnb_dijkstra_batch_sharded", "mnb_cvp_batch_sharded",
              "mnb_group_read_fields", "mnb_group_read_preds"):
        getattr(L, f).restype = C.c_int32
    L.mnb_group_row.restype = C.c_uint32; L.mnb_group_size.restype = C.c_int32; L.mnb_group_last_error.restype = C.c_char_p
    L.mnb_group_preds.restype = C.c_void_p; L.mnb_group_preds.argtypes = [C.c_void_p, C.c_int32]
    L.mnb_dijkstra_batch_sharded.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_double, C.c_int32, C.c_int32]
    L.mnb_cvp_batch_sharded.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_double, C.c_int32]
    L.mnb_group_read_fields.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_uint32, C.c_void_p]
    L.mnb_group_read_preds.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_uint32, C.c_void_p]
    L.mnb_group_set_mesh.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
    L.mnb_group_set_costs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mnb_group_row.argtypes = [C.c_void_p, C.c_uint32]; L.mnb_group_size.argtypes = [C.c_void_p]; L.mnb_group_destroy.argtypes = [C.c_void_p]
    L.mnb_group_last_error.argtypes = [C.c_void_p]
    devs = (C.c_int32 * ndev)(*range(ndev)); grp = C.c_void_p()
    assert L.mnb_group_create(ndev, devs, C.byref(grp)) == 0 and L.mnb_group_size(grp) == ndev
    assert L.mnb_dijkstra_batch_sharded(grp, 1, p(np.zeros(1, np.uint32)), 1.0, 1, 1) == -3      # MNB_E_STATE: no map yet
    edges = np.ascontiguousarray(om.edges, np.uint32)
    assert L.mnb_group_set_mesh(grp, om.V, om.F, p(pos), p(faces), p(edges), edges.shape[0]) == 0
    assert L.mnb_group_set_costs(grp, p(vc), p(ed), None) == 0
    n = 7                                                                   # ragged: ranks own 4 and 3 goals
    seeds = np.random.default_rng(4).integers(0, om.V, n).astype(np.uint32)
    assert L.mnb_dijkstra_batch_sharded(grp, n, p(seeds), 1.0, 1, 1) == 0, L.mnb_group_last_error(grp)
    pad = (n + ndev - 1) // ndev
    assert [L.mnb_group_row(grp, k) for k in range(n)] == [(k % ndev) * pad + k // ndev for k in range(n)]
    refs = [om.dijkstra(ed, vc, int(s)) for s in seeds]
    for rank in range(ndev):                                                # every rank holds every field and pred row
        assert L.mnb_group_preds(grp, rank)
        dist = np.empty((n, om.V), np.float32); pred = np.empty((n, om.V), np.uint32)
        assert L.mnb_group_read_fields(grp, rank, 0, n, p(dist)) == 0
        assert L.mnb_group_read_preds(grp, rank, 0, n, p(pred)) == 0
        for k in range(n):
            assert (dist[k].view(np.uint32) == refs[k]["dist"].view(np.uint32)).all(), (rank, k)
            assert (pred[k] == refs[k]["pred"]).all(), (rank, k)
    # without want_pred, and after a CVP sharded call, there are no predecessors to read
    out = np.empty((1, om.V), np.uint32)
    assert L.mnb_dijkstra_batch_sharded(grp, n, p(seeds), 1.0, 0, 1) == 0
    assert L.mnb_group_read_preds(grp, 0, 0, 1, p(out)) == -3
    assert L.mnb_dijkstra_batch_sharded(grp, n, p(seeds), 1.0, 1, 1) == 0
    sfs = np.array([1, 2], np.uint32); sps = np.stack([pos[faces[f]].mean(0) for f in sfs]).astype(np.float32)
    assert L.mnb_cvp_batch_sharded(grp, 2, p(sfs), p(sps), 1.0, 1) == 0
    assert L.mnb_group_read_preds(grp, 0, 0, 1, p(out)) == -3
    L.mnb_group_destroy(grp)
