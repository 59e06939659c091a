#!/usr/bin/env python
"""bench.py -- headline measurement of the wavefront hot path (contract in the task brief).

step      = one full-field CVP plan (CVPMeshPlanner::waveFrontPropagation, no goal cutoff) per GPU
            on the 5M-vertex synthetic terrain mesh (2240 x 2240, SURVEY.md 8d); with N GPUs every
            rank plans a different goal on its replica of the map (one-goal-per-GPU sharding) and
            the potential arrays are all-gathered over NCCL inside the timed region.
value     = settled vertices of all ranks / device time, inputs already resident in HBM.
e2e       = same plan through the C ABI with HOST buffers: vertex_costs + edge_weights copied H2D
            (mnb_set_costs) and potential/pred/direction/cutting_face copied D2H every step.
roofline  = dominant kernel k_cvp: algorithmic bytes (208 B / settled vertex, SURVEY.md 8d) / its
            CUDA-event duration, against the measured HBM copy bandwidth (MEASURED_PEAKS.json).
cpu_baseline = the oracle (reference algorithm restated, 1 thread, as the reference is per plan), rebuilt on the box
            with -O3 -march=native (BASELINE.md section 2).
config.parity    = the potentials / predecessors of the TIMED 5M plan against the oracle's plan on the same input
                   (canonical ties); a deviation above 1e-4 fails the run (exit code 3 after the line is printed).
config.config3   = BASELINE config 3 as a plan: fused layers -> Max combination with the inflation of (layer lethals +
                   1000 obstacle discs) -> vertex_costs -> computeEdgeWeights(edge_cost_factor 1) -> CVP with
                   cost_limit 1 on those costs, timed, with its own parity block.
config.batched   = BASELINE config 4 (1024 goals, 1M-vertex terrain, goal k -> rank k mod N, potentials all-gathered):
                   plans/s, HBM fraction and 8 sampled fields against the oracle -- inside `config` because the driver
                   keeps that object for every N.
--impl reference: the oracle on the host cores, one independent plan per thread.
--dump-outputs DIR: the arrays the last timed plan returned, as DIR/<name>.npy (dump_outputs()); the inputs are seeded, so
                   two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

CVP_BYTES_PER_VERTEX = 208       # SURVEY.md 8d
METRIC = "vertex-relaxations/sec"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    def __init__(self):
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
                 "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self, device=0):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9 or f[0] != str(device):
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(workload):
    """dram bytes (read + write) per launch of the dominant kernel from the committed `ncu --set full` capture"""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


def build_workload(n):
    from mesh_navigation_b200 import synth
    pos, faces = synth.grid_mesh(n, n, terrain=True, seed=42)
    return pos, faces


def goal_for_rank(pos, faces, n, rank):
    """rank 0: face at the map centre (SURVEY 8d config 2); other ranks: distinct goals within 2 % of the map size around
    the centre, so that every GPU solves a wave of the same depth (weak scaling: per-GPU work fixed)."""
    from mesh_navigation_b200 import synth
    offs = [(0, 0), (1, 1), (-1, 1), (1, -1), (-1, -1), (1, 0), (-1, 0), (0, 1)]
    ox, oy = offs[rank % len(offs)]
    d = 0.02 * n * 0.1 * (1 + rank // len(offs))
    v = synth.nearest_vertex(pos, [n * 0.05 + ox * d, n * 0.05 + oy * d, float(pos[:, 2].mean())])
    i, j = v % n, v // n
    i = min(i, n - 2); j = min(j, n - 2)
    f = 2 * (j * (n - 1) + i)
    return f, pos[faces[f]].mean(0).astype(np.float32)


def parity_block(got_dist, got_pred, ref, got_cut=None):
    """GPU plan against the oracle plan of the same input: bit mismatches, largest relative deviation, predecessor /
    cutting-face mismatches (north star: potentials within 1e-4 rel, indices exact)"""
    gd, rd = np.asarray(got_dist), ref["dist"]
    fin = np.isfinite(rd)
    same_set = bool(np.array_equal(np.isfinite(gd), fin))
    rel = np.abs(gd[fin] - rd[fin]) / np.maximum(rd[fin], 1e-30) if same_set else np.array([np.inf])
    out = {"vertices_compared": int(rd.size), "reached_sets_equal": same_set,
           "n_mismatch": int((gd.view(np.uint32) != rd.view(np.uint32)).sum()), "max_rel": float(rel.max()) if rel.size else 0.0,
           "pred_mismatch": None if got_pred is None else int((np.asarray(got_pred).astype(np.int64) != ref["pred"].astype(np.int64)).sum())}
    if got_cut is not None:
        out["cutting_face_mismatch"] = int((np.asarray(got_cut).astype(np.int64) != ref["cutting_face"].astype(np.int64)).sum())
    out["ok"] = bool(same_set and out["max_rel"] <= 1e-4 and not out["pred_mismatch"])
    return out


DUMP_MAX_VERTICES = 1 << 20     # 32 B per dumped vertex (two f32, three f64 arrays): at most 32 MiB in all


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the per-vertex arrays a caller of the timed plan receives (potential, predecessor, direction, cutting
    face), so that two builds can be compared output for output.  Above DUMP_MAX_VERTICES vertices a fixed, seeded sample
    of vertices is written; vertex_index.npy names them.  Float arrays stay float32, index arrays become float64 (exact)."""
    V = next(iter(arrays.values())).size
    idx = np.arange(V) if V <= DUMP_MAX_VERTICES else np.sort(np.random.default_rng(0).choice(V, DUMP_MAX_VERTICES, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "vertex_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[idx].astype(np.float32 if a.dtype.kind == "f" else np.float64))


CONFIG_KEYS = ("workload", "vertices", "faces", "edges", "plans_per_step_per_gpu", "sharding", "l2", "parity", "config3", "batched")


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; lvr2 / ROS 2 cannot be installed offline)
    on the host cores, on the SAME workload as the B200 arm: one full-field CVP plan on the 5M-vertex terrain per
    step.  The reference plans one query on one thread (MeshPlannerExecution::makePlan runs the heap loop on the
    planner thread, mesh_planner_execution.cpp:55-66), so a single plan uses 1 core; the batched sub-result uses
    one independent plan per host thread on all cores (BASELINE.md section 2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    flags = O.use_native_build()             # -O3 -march=native, built on this host (BASELINE.md section 2)
    n = args.size
    pos, faces = build_workload(n)
    om = O.OracleMesh(pos, faces)
    ed = om.edge_distances(); vc = np.zeros(om.V, np.float32)
    sf, sp = goal_for_rank(pos, faces, n, 0)
    settled = 0

    def step():
        nonlocal settled
        r = om.cvp(ed, vc, sf, sp, canonical_ties=False)      # plain lvr2-style heap
        settled = int(np.isfinite(r["dist"]).sum())
        return r["seconds"]

    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter(); prop = 0.0
    for _ in range(args.steps):
        prop += step()
    dt = time.perf_counter() - t0
    value = settled * args.steps / prop                        # propagation phase only, like the reference's own log line
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "vertices/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * prop / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 update / f32 store", "data": "synthetic",
        "config": {"workload": f"cvp_full_field_terrain_{n}x{n}", "vertices": om.V, "faces": om.F, "edges": om.E,
                   "plans_per_step_per_gpu": 1,
                   "sharding": "host CPU, one thread per plan (the reference's loop is single-threaded per plan, mesh_planner_execution.cpp:55-66)",
                   "l2": "n/a (CPU); timed region = heap loop (cvp_mesh_planner.cpp:744-894), wall per step "
                         f"{1e3 * dt / args.steps:.0f} ms incl. array init",
                   "parity": None, "config3": None, "batched": None},
        "cpu_baseline": {"value": value, "unit": "vertices/s", "cores": 1, "kind": "port", "flags": flags,
                         "sample": f"{args.steps} full-field plans on the {n}x{n} terrain; the reference's loop is single-threaded per plan"},
        "e2e": {"value": value, "unit": "vertices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    # batched: one independent plan per host thread (config 4 shape, bounded sample)
    if args.batch_goals > 0:
        nb = args.batch_size
        bpos, bfaces = build_workload(nb)
        bom = O.OracleMesh(bpos, bfaces)
        bed = bom.edge_distances(); bvc = np.zeros(bom.V, np.float32)
        cores = os.cpu_count() or 1
        nthreads = max(1, min(cores, args.ref_threads))
        goals = [goal_for_rank(bpos, bfaces, nb, r % 60) for r in range(nthreads)]

        def work(i):
            bom.cvp(bed, bvc, goals[i][0], goals[i][1], canonical_ties=False)

        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(i,)) for i in range(nthreads)]
        [t.start() for t in th]; [t.join() for t in th]
        dtb = time.perf_counter() - t0
        line["config"]["batched"] = {"plans_per_s": nthreads / dtb, "goals": nthreads, "mesh_vertices": int(bom.V), "cores": nthreads,
                                     "vertex_relaxations_per_s": nthreads * bom.V / dtb, "ms_per_batch": 1e3 * dtb,
                                     "sample": f"{nthreads} concurrent full-field plans (one per host thread, {cores} logical cores) on the {nb}x{nb} terrain"}
        line["batched"] = line["config"]["batched"]
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=2240, help="grid side (2240 -> 5,017,600 vertices)")
    ap.add_argument("--ref-size", type=int, default=1000, help="grid side of the CPU reference sample")
    ap.add_argument("--ref-threads", type=int, default=64)
    ap.add_argument("--cluster", type=int, default=0)
    ap.add_argument("--delta", type=float, default=0.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--batch-goals", type=int, default=1024, help="goals of the batched leg (config 4); 0 disables it")
    ap.add_argument("--batch-size", type=int, default=1000, help="grid side of the batched leg's mesh")
    ap.add_argument("--batch-steps", type=int, default=2)
    ap.add_argument("--batch-delta", type=float, default=0.0, help="band width of the batched leg (0 = library default)")
    ap.add_argument("--batch-cluster", type=int, default=0, help="CTAs per wavefront of the batched leg (0 = chosen per call)")
    ap.add_argument("--no-config3", action="store_true")
    ap.add_argument("--no-other-kernels", action="store_true")
    ap.add_argument("--submesh-from", type=int, default=3000, help="grid side from which the 1M sub-mesh parity spot check runs (config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed plan returned (rank 0) to DIR/<name>.npy, see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from mesh_navigation_b200.api import MeshMap

    n = args.size
    pos, faces = build_workload(n)
    mm = MeshMap(pos, faces, device=local)
    if args.cluster or args.delta:
        mm.set_tuning(args.delta, args.cluster, 0)
    V, E = mm.V, mm.E
    ed = mm.edgeDistances()
    vc = np.zeros(V, np.float32)
    mm.setCosts(vc, ed)
    sf, sp = goal_for_rank(pos, faces, n, rank)
    dev = torch.device("cuda", local)
    d_dist = torch.empty(V, dtype=torch.float32, device=dev)
    d_pred = torch.empty(V, dtype=torch.int32, device=dev)
    d_dir = torch.empty(V, dtype=torch.float32, device=dev)
    d_cut = torch.empty(V, dtype=torch.int32, device=dev)
    gathered = [torch.empty(V, dtype=torch.float32, device=dev) for _ in range(world)] if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2

    def step_resident():
        flush.zero_()                                   # L2 flush between timed iterations (untimed kernels are tiny)
        mm.use_device_pointers(True)
        mm.cvp_dev(sf, sp, -1, 1.0, 0.3, d_dist.data_ptr(), d_pred.data_ptr(), d_dir.data_ptr(), d_cut.data_ptr())
        mm.use_device_pointers(False)
        st = mm.stats()
        if world > 1:
            dist.all_gather(gathered, d_dist)
        return st

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident()
    sync_all()
    sampler = ClockSampler(); sampler.start()
    kernel_ms, settled = [], 0
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = step_resident()              # mnb_cvp returns after the stream drained (stats read back)
        kernel_ms.append(st["kernel_ms"]); settled = st["settled"] + 3
    sync_all()
    dt = time.perf_counter() - t0
    # device-side time of the timed region = sum of the CUDA-event bracketed kernels (+ gather for N>1 is in dt)
    t = torch.tensor([dt, float(settled)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dt_max = float(tmax[0]); total_settled = float(tsum[1])
    else:
        dt_max = dt; total_settled = float(settled)
    clocks = sampler.stop(local)
    value = total_settled * args.steps / dt_max
    # the result of the LAST TIMED plan, for the parity block and the output dump (rank 0)
    h_timed = None
    if rank == 0 and (not args.no_cpu_baseline or args.dump_outputs):
        h_timed = {"dist": d_dist.cpu().numpy(), "pred": d_pred.cpu().numpy().view(np.uint32), "cut": d_cut.cpu().numpy()}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"dist": h_timed["dist"], "pred": h_timed["pred"], "direction": d_dir.cpu().numpy(),
                                             "cutting_face": h_timed["cut"]})

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ----
    from mesh_navigation_b200.api import CVPMeshPlanner
    planner = CVPMeshPlanner(mm)
    # pinned host buffers for the per-step inputs (vertex_costs, edge_weights) and outputs
    pin = lambda nelem, dt: torch.empty(nelem, dtype=dt).pin_memory().numpy()
    h_vc = pin(V, torch.float32); h_vc[:] = 0.0
    h_ew = pin(E, torch.float32); h_ew[:] = ed
    h_out = {"dist": pin(V, torch.float32), "pred": pin(V, torch.int32).view(np.uint32),
             "direction": pin(V, torch.float32), "cutting_face": pin(V, torch.int32)}
    e2e_steps = max(2, args.steps // 2)
    for _ in range(2):
        mm.setCosts(h_vc, h_ew); planner.waveFrontPropagation(sf, sp, out=h_out)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        mm.setCosts(h_vc, h_ew)
        out = planner.waveFrontPropagation(sf, sp, out=h_out)
        if world > 1:
            d_dist.copy_(torch.from_numpy(out["dist"])); dist.all_gather(gathered, d_dist)
    sync_all()
    dte = time.perf_counter() - t0
    te = torch.tensor([dte], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total_settled * e2e_steps / float(te[0])

    # ---- batched leg (config 4): G goals on the 1M terrain, goal k -> rank k mod N, potentials all-gathered ----
    batched = None
    if args.batch_goals > 0:
      try:
          from mesh_navigation_b200 import parallel as PL
          from mesh_navigation_b200 import synth
          nb = args.batch_size
          bpos, bfaces = build_workload(nb)
          bm = MeshMap(bpos, bfaces, device=local)
          bed = bm.edgeDistances()
          bm.setCosts(np.zeros(bm.V, np.float32), bed)
          if args.batch_delta > 0 or args.batch_cluster:
              bm.set_tuning(args.batch_delta, args.batch_cluster, 0)
          goals = synth.batch_goal_vertices(bm.V, args.batch_goals, seed=1234)
          gi, gj = np.minimum(goals % nb, nb - 2), np.minimum(goals // nb, nb - 2)
          sfs = (2 * (gj * (nb - 1) + gi)).astype(np.uint32)
          sps = bpos[bfaces[sfs]].mean(1).astype(np.float32)
          bm.use_device_pointers(True)
          b_kernel_ms, b_gather_ms = [], []

          def compute_chunk(idx, out):
              bm.cvp_batch_dev(sfs[idx], sps[idx], 1.0, out.data_ptr())
              b_kernel_ms.append(bm.stats()["kernel_ms"])

          def batch_step():
              tm = {}
              res = PL.sharded_potentials(compute_chunk, args.batch_goals, bm.V, rank=rank, world=world, device=dev,
                                          chunk=0, dist=dist if world > 1 else None, torch=torch, timings=tm)
              b_gather_ms.append(tm.get("gather_ms", 0.0))
              return res

          res = batch_step(); sync_all()
          b_kernel_ms.clear(); b_gather_ms.clear()
          t0 = time.perf_counter()
          for _ in range(args.batch_steps):
              del res
              res = batch_step()
          sync_all()
          dtb = time.perf_counter() - t0
          tb = torch.tensor([dtb, sum(b_kernel_ms), sum(b_gather_ms)], dtype=torch.float64, device=dev)
          if world > 1:
              dist.all_reduce(tb, op=dist.ReduceOp.MAX)
          dtb = float(tb[0])
          bm.use_device_pointers(False)
          plans_s = args.batch_goals * args.batch_steps / dtb
          my_goals = len(PL.shard_indices(args.batch_goals, rank, world))
          b_achieved = CVP_BYTES_PER_VERTEX * bm.V * my_goals * args.batch_steps / (sum(b_kernel_ms) * 1e-3) / 1e9
          batched = {"plans_per_s": plans_s, "goals": args.batch_goals, "goals_per_gpu": my_goals, "mesh_vertices": int(bm.V), "n_gpus": world,
                     "vertex_relaxations_per_s": plans_s * bm.V, "ms_per_batch": 1e3 * dtb / args.batch_steps,
                     "compute_ms_per_batch_max_rank": float(tb[1]) / args.batch_steps, "gather_ms_per_batch_max_rank": float(tb[2]) / args.batch_steps,
                     "scaling": "strong (fixed goal count)",
                     "gather": "one NCCL all_gather_into_tensor of float[goals][V] into the final buffer after the rank's batch call" if world > 1 else "none (single GPU)",
                     "roofline_hbm_frac_rank0": b_achieved / peaks()[0], "achieved_gbs_rank0": b_achieved,
                     "recomputes_per_vertex": bm.stats()["recomputes"] / max(1, my_goals) / bm.V}
          if rank == 0 and not args.no_cpu_baseline:
              # 8 of the fields against the oracle (every rank's shard is covered: the gathered buffer is in goal order)
              from oracle import oracle as O
              bom = O.OracleMesh(bpos, bfaces)
              bvc = np.zeros(bm.V, np.float32)
              rows = PL.goal_order_rows(res, args.batch_goals, bm.V) if world > 1 else res
              samp = np.unique(np.linspace(0, args.batch_goals - 1, 8).astype(np.int64))
              worst, nmis = 0.0, 0
              for k in samp:
                  pb = parity_block(rows[int(k)].cpu().numpy(), None, bom.cvp(bed, bvc, int(sfs[k]), sps[k]))
                  worst = max(worst, pb["max_rel"]); nmis += pb["n_mismatch"]
              batched["parity_sampled"] = {"fields": [int(k) for k in samp], "n_mismatch": int(nmis), "max_rel": worst, "ok": bool(worst <= 1e-4)}
          del res
          bm.close()
      except Exception as ex:      # a secondary leg must never cost the headline line (all ranks fail alike: no collective is left half-done)
        batched = {"error": f"{type(ex).__name__}: {ex}"}

    # ---- the other hot-path kernels on the same mesh (rank 0, one run each after a warm-up; SURVEY 8a rows a1/a7/a10 + f1/f2) ----
    other = None
    if rank == 0 and not args.no_other_kernels:
        from mesh_navigation_b200 import synth
        from mesh_navigation_b200.api import DijkstraMeshPlanner, InflationLayer
        hbm0 = peaks()[0]
        other = {}
        shared = {}

        def leg(name, fn):               # a secondary leg must never cost the headline line
            try:
                other[name] = fn()
            except Exception as ex:
                other[name] = {"error": f"{type(ex).__name__}: {ex}"}

        def leg_dijkstra():
            seed_v = int(faces[sf][0])
            for rep in range(2):
                D = DijkstraMeshPlanner(mm).dijkstra(seed_v)
            return {"kernel_ms": D["kernel_ms"], "rounds": int(D["rounds"]), "vertices_per_s": V / (D["kernel_ms"] * 1e-3),
                    "hbm_frac": 92 * V / (D["kernel_ms"] * 1e-3) / 1e9 / hbm0}

        def leg_layers():
            for rep in range(2):
                Ly = mm.computeLayers()
            shared["lethal_mask"] = Ly["lethal_mask"]; shared["combined"] = Ly["combined"]; shared["layers_ms"] = Ly["kernel_ms"]
            return {"kernel_ms": Ly["kernel_ms"], "hbm_frac": 837 * V / (Ly["kernel_ms"] * 1e-3) / 1e9 / hbm0}

        def leg_inflation():
            n_discs = max(2, int(round(1000 * (n / 2240.0) ** 2)))         # 1000 obstacle discs on the 5M map, same density on smaller ones
            le = np.union1d(np.where(shared["lethal_mask"] != 0)[0], synth.disc_lethals_grid(pos, n, n, n_discs, 0.3)).astype(np.uint32)
            shared["lethals"] = le
            for rep in range(2):
                I = InflationLayer(mm).waveCostInflation(le)
            nin = int(np.isfinite(I["dist"]).sum())
            return {"kernel_ms": I["kernel_ms"], "rounds": int(I["rounds"]), "lethal_vertices": int(le.size), "labelled_vertices": nin,
                    "hbm_frac": 212 * nin / (I["kernel_ms"] * 1e-3) / 1e9 / hbm0}

        def leg_config3():
            """BASELINE config 3 as a PLAN on the 5M map (mesh_map.cpp:437-448,539-553; inflation_layer.cpp:563-596): the
            layer stack's costs (fused layers, Max-combined with the inflation of layer lethals + 1000 obstacle discs)
            become vertex_costs, computeEdgeWeights(edge_cost_factor 1) the planner's weights, and a full-field CVP plan
            with cost_limit 1 runs on them -- lethal walls, cost-weighted non-geometric weights, back-steps, cascades"""
            static = shared["combined"]; le = shared["lethals"]
            infl = InflationLayer(mm)
            I = infl.waveCostInflation(le)
            final = np.maximum(static, np.nan_to_num(I["cost"], nan=0.0)).astype(np.float32)    # MaxCombinationLayer, defaults 0
            t0 = time.perf_counter(); w1 = mm.computeEdgeWeights(final, 1.0); t_w = time.perf_counter() - t0
            free = np.where(final < 0.5)[0]
            if free.size == 0:
                free = np.argsort(final)[:16]
            c0 = synth.nearest_vertex(pos, [n * 0.05, n * 0.05, float(pos[:, 2].mean())])
            v = int(free[np.argmin(np.linalg.norm(pos[free] - pos[c0], axis=1))])
            i, j = min(v % n, n - 2), min(v // n, n - 2)
            f = 2 * (j * (n - 1) + i)
            while not (final[faces[f]] < 1.0).all() and f + 1 < mm.F:
                f += 1
            spc = pos[faces[f]].mean(0).astype(np.float32)
            pl3 = CVPMeshPlanner(mm, cost_limit=1.0)
            best = None
            for rep in range(3):
                g = pl3.waveFrontPropagation(f, spc)
                best = g["kernel_ms"] if best is None else min(best, g["kernel_ms"])
            reached = int(np.isfinite(g["dist"]).sum())
            out = {"stages_ms": {"fused_layers_kernel": shared.get("layers_ms"), "inflation_kernel": I["kernel_ms"], "edge_weights_wall": 1e3 * t_w, "cvp_kernel": best},
                   "kernel_ms": best, "reached_vertices": reached, "vertices_per_s": reached / (best * 1e-3),
                   "hbm_frac": CVP_BYTES_PER_VERTEX * reached / (best * 1e-3) / 1e9 / hbm0,
                   "lethal_vertices": int((final >= 1.0).sum()), "rounds": int(g["rounds"]), "recomputes_per_vertex": g["recomputes"] / max(1, reached),
                   "deep_cascade_labels": int(g.get("deep_labels", 0)), "level_pool_words": int(g.get("pool_words", 0)), "outcome": int(g["outcome"])}
            if not args.no_cpu_baseline:
                from oracle import oracle as O
                om3 = O.OracleMesh(pos, faces)
                wref = om3.edge_weights(final, ed, 1.0)
                ref3 = om3.cvp(wref, final, f, spc, cost_limit=1.0)
                pb = parity_block(g["dist"], g["pred"], ref3, g["cutting_face"])
                pb["edge_weights_bit_identical"] = bool((w1.view(np.uint32) == wref.view(np.uint32)).all())
                refi = om3.inflation(ed, le)
                pb["inflation_dist_mismatch"] = int((I["dist"].view(np.uint32) != refi["dist"].view(np.uint32)).sum())
                pb["oracle_backsteps"] = int(ref3["backsteps"]); pb["oracle_cvp_seconds"] = float(ref3["seconds"])
                out["parity"] = pb
            mm.setCosts(vc, ed)
            return out

        def leg_dynamic_update():
            """one dynamic-obstacle cycle (SURVEY 3.4) on the 5M map with every array resident on the device (MNB_PTR_DEVICE,
            torch tensors): the 1000 discs move; InflationLayer::onInputChanged -> MaxCombinationLayer::onInputChanged on the
            update set -> MeshMap::layerChanged (incremental: only the table entries of the incident edges are patched), wall
            times around torch.cuda.synchronize(); the resulting tables are compared with a full re-install"""
            import ctypes as C
            infl = InflationLayer(mm)
            static = shared["combined"]
            base = np.where(shared["lethal_mask"] != 0)[0]
            n_discs = max(2, int(round(1000 * (n / 2240.0) ** 2)))
            le0 = np.union1d(base, synth.disc_lethals_grid(pos, n, n, n_discs, 0.3, seed=7)).astype(np.uint32)
            le1 = np.union1d(base, synth.disc_lethals_grid(pos, n, n, n_discs, 0.3, seed=8)).astype(np.uint32)
            r0 = infl.onInputChanged(le0)
            final0 = np.maximum(static, np.nan_to_num(r0["cost"], nan=0.0)).astype(np.float32)
            mm.computeEdgeWeights(final0, 1.0, want_output=False)
            d_static = torch.from_numpy(static).to(dev); d_final = torch.from_numpy(final0).to(dev)
            d_le = [torch.from_numpy(x.astype(np.int64)).to(dev).to(torch.int32) for x in (le1, le0)]
            d_dist = torch.empty(V, dtype=torch.float32, device=dev); d_cost = torch.empty(V, dtype=torch.float32, device=dev)
            d_changed = torch.empty(V, dtype=torch.int32, device=dev); d_vec = torch.empty((V, 3), dtype=torch.float32, device=dev)
            p = lambda t: C.c_void_p(t.data_ptr())
            nch = C.c_uint32(0); defaults = np.zeros(2, np.float32); Lc = mm.L; cx = mm._ctx
            mm.use_device_pointers(True)

            def cycle(k, with_field):
                t = {}
                torch.cuda.synchronize(); t0 = time.perf_counter()
                assert Lc.mnb_inflation_update(cx, p(d_le[k]), int(d_le[k].numel()), None, C.byref(infl.config), p(d_dist), p(d_cost), p(d_changed), C.byref(nch)) == 0
                torch.cuda.synchronize(); t1 = time.perf_counter(); t["inflation_update_ms"] = 1e3 * (t1 - t0); t["inflation_kernel_ms"] = mm.stats()["kernel_ms"]
                lc = (C.c_void_p * 2)(d_static.data_ptr(), d_cost.data_ptr())
                assert Lc.mnb_max_combination_update(cx, 2, lc, defaults.ctypes.data_as(C.c_void_p), None, nch.value, p(d_changed), p(d_final), None) == 0
                torch.cuda.synchronize(); t2 = time.perf_counter(); t["max_combination_ms"] = 1e3 * (t2 - t1)
                assert Lc.mnb_update_vertex_costs(cx, nch.value, p(d_changed), p(d_final), 1, 0.0, 1.0) == 0
                torch.cuda.synchronize(); t3 = time.perf_counter(); t["layer_changed_ms"] = 1e3 * (t3 - t2)
                t["total_wall_ms"] = 1e3 * (t3 - t0)
                if with_field:
                    assert Lc.mnb_inflation_vector_map(cx, p(d_vec)) == 0
                    torch.cuda.synchronize(); t["repulsive_vector_field_ms"] = 1e3 * (time.perf_counter() - t3)
                return t

            try:
                for rep in range(2):
                    cycle(0, False); cycle(1, False)
                ta = cycle(0, True)
            finally:
                mm.use_device_pointers(False)
            gvc, gw = mm.costs()
            final1 = d_final.cpu().numpy()
            full_w = mm.computeEdgeWeights(final1, 1.0)
            ref1 = np.maximum(static, np.nan_to_num(infl.onInputChanged(le1)["cost"], nan=0.0)).astype(np.float32)
            same = bool((gw.view(np.uint32) == full_w.view(np.uint32)).all() and (gvc.view(np.uint32) == final1.view(np.uint32)).all()
                        and (final1.view(np.uint32) == ref1.view(np.uint32)).all())
            mm.setCosts(vc, ed)
            ta.update({"changed_vertices": int(nch.value), "lethal_vertices": int(le1.size), "incremental_equals_full": same,
                       "arrays": "device-resident (MNB_PTR_DEVICE); the update set and its size are produced on the device, only the count is read back"})
            return ta

        def leg_submesh_parity():
            """BASELINE.md row 5: parity spot check on a 1M-vertex sub-mesh of the large terrain -- the 1000x1000 window of the
            same vertices around the goal is cut out, installed as its own map, and layers + a full-field CVP plan on it
            are compared bit for bit with the oracle"""
            from oracle import oracle as O
            m = min(1000, n // 2)
            v0 = int(faces[sf][0]); i0 = min(max(v0 % n - m // 2, 0), n - m); j0 = min(max(v0 // n - m // 2, 0), n - m)
            spos = np.ascontiguousarray(pos.reshape(n, n, 3)[j0:j0 + m, i0:i0 + m].reshape(-1, 3))
            sfaces = synth.grid_mesh(m, m)[1]
            sm = MeshMap(spos, sfaces, device=local)
            try:
                sed = sm.edgeDistances(); svc = np.zeros(sm.V, np.float32); sm.setCosts(svc, sed)
                fi, fj = v0 % n - i0, v0 // n - j0
                f = 2 * (min(fj, m - 2) * (m - 1) + min(fi, m - 2)); spc = spos[sfaces[f]].mean(0).astype(np.float32)
                g = CVPMeshPlanner(sm).waveFrontPropagation(f, spc)
                Ly = sm.computeLayers()
                som = O.OracleMesh(spos, sfaces)
                ref = som.cvp(som.edge_distances(), svc, f, spc)
                out = {"window": [int(i0), int(j0), m, m], "vertices": int(sm.V), "cvp": parity_block(g["dist"], g["pred"], ref, g["cutting_face"])}
                rl = som.layers()
                out["layers_bit_mismatch"] = {k: int((Ly[k].view(np.uint32) != rl[k].view(np.uint32)).sum()) for k in ("height_diff", "ridge", "border", "roughness", "steepness")}
                rel = max(float(np.max(np.abs(Ly[k] - rl[k]) / np.maximum(np.abs(rl[k]), 1e-30))) for k in ("roughness", "steepness"))
                out["layers_acos_max_rel"] = rel           # double acos, rounded once on both sides: last-bit differences only
                out["lethal_masks_identical"] = bool((Ly["lethal_mask"] == rl["lethal_mask"]).all())
                out["ok"] = bool(out["cvp"]["ok"] and out["lethal_masks_identical"] and rel <= 2e-7
                                 and not any(out["layers_bit_mismatch"][k] for k in ("height_diff", "ridge", "border")))
            finally:
                sm.close()
            return out

        def leg_obstacle_raycast():
            """the input side of the dynamic cycle (SURVEY 8 f3): a 262 144-point cloud through ObstacleLayer::processPointCloud
            (obstacle_layer.cpp:215-296) on the bench map -- BVH build (once per map), range filter + transform + one ray per
            point + lethal / changed sets; then calcNormalClearance (one ray per vertex).  Parity: a sample of the rays against
            the oracle's loop over all faces"""
            from mesh_navigation_b200.api import ObstacleLayer
            rng = np.random.default_rng(5)
            npts = 262144 if n >= 1000 else 2048
            c = pos[(n // 2) * n + n // 2]
            ij = rng.integers(0, n, size=(npts, 2))
            base = pos[ij[:, 1] * n + ij[:, 0]]
            near = np.linalg.norm(base[:, :2] - c[:2], axis=1) <= 12.0 if n >= 1000 else np.ones(npts, bool)
            ij2 = np.clip(((c[:2] / 0.1)[None, :] + rng.normal(size=(npts, 2)) * 40.0).astype(np.int64), 0, n - 1)
            base = np.where(near[:, None], base, pos[ij2[:, 1] * n + ij2[:, 0]])
            pts_map = (base + np.stack([rng.normal(size=npts) * 0.02, rng.normal(size=npts) * 0.02, rng.random(npts) * 1.5 + 0.02], 1)).astype(np.float32)
            pts = (pts_map - c).astype(np.float32)                                    # message frame: origin at the robot
            T = np.hstack([np.eye(3, dtype=np.float32), c.reshape(3, 1)]).astype(np.float32)
            t0 = time.perf_counter(); layer = ObstacleLayer(mm, robot_height=1.0, max_obstacle_dist=10.0)
            mm.castRays(pts_map[:4], np.array([0, 0, -1], np.float32)); t_build = time.perf_counter() - t0
            for rep in range(2):
                t0 = time.perf_counter(); r = layer.processPointCloud(pts, T); t_wall = time.perf_counter() - t0
            out = {"points": npts, "bvh_build_wall_ms": 1e3 * t_build, "faces": int(mm.F), "process_point_cloud_wall_ms": 1e3 * t_wall,
                   "process_point_cloud_kernels_ms": r["kernel_ms"], "lethal_vertices": int(r["lethals"].size),
                   "rays_per_s": npts / (r["kernel_ms"] * 1e-3)}
            t0 = time.perf_counter(); cl = mm.normalClearance(); out["normal_clearance_wall_ms"] = 1e3 * (time.perf_counter() - t0)
            out["normal_clearance_kernel_ms"] = mm.stats()["kernel_ms"]; out["finite_clearances"] = int(np.isfinite(cl).sum())
            if not args.no_cpu_baseline:
                from oracle import oracle as O
                om = O.OracleMesh(pos, faces)
                k = min(128 if mm.F < 1000000 else 32, npts)        # the oracle visits every face for every ray
                down = np.array([0, 0, -1], np.float32)
                got = mm.castRays(pts_map[:k], down); t0 = time.perf_counter(); ref = om.cast_rays(pts_map[:k], down); t_or = time.perf_counter() - t0
                out["parity_sampled"] = {"rays": k, "ok": bool((got["face"] == ref["face"]).all() and (got["dist"].view(np.uint32) == ref["dist"].view(np.uint32)).all()
                                                               and (got["hit"] == ref["hit"]).all()),
                                         "oracle_rays_per_s": k / t_or}
            return out

        def leg_make_plan():
            # a whole makePlan through the host API: localisation of both poses, wavefront until the robot face is fixed,
            # vector-field back-tracking on the device; only the path crosses PCIe
            corner = lambda u, v: pos[int(v * (n - 1)) * n + int(u * (n - 1))]
            pts = np.stack([corner(0.1, 0.1), corner(0.9, 0.9)]).astype(np.float32)
            mm.setCosts(vc, ed)
            for rep in range(2):
                t0 = time.perf_counter()
                nv, fc, ba = mm.locate(pts)
                mp = planner.makePlan(pts[0], int(fc[0]), pts[1], int(fc[1]))
                tmp = time.perf_counter() - t0
            return {"wall_ms": 1e3 * tmp, "wavefront_kernel_ms": mp.get("wavefront_ms"), "path_points": int(len(mp["positions"])),
                    "path_length_m": mp["cost"], "outcome": int(mp["outcome"])}

        def leg_optin_variants():
            """A/B of the opt-in kernel variants that were written and verified on the CPU interpreter of the kernels after the
            round's GPU budget was spent (DESIGN.md 4/5/9): each is run next to the default kernel on the bench mesh and
            compared bit for bit.  Run last: nothing above depends on them."""
            import ctypes as C
            out = {}
            for f in ("mnb_debug_set_layers_smem", "mnb_debug_set_infl_skip"):
                getattr(mm.L, f).argtypes = [C.c_void_p, C.c_int32]
            # the inflation wave's clean-candidate skip is ON by default: time it against the all-candidates-every-round loop
            le = shared.get("lethals")
            if le is not None:
                res = {}
                for on in (1, 0, 1, 0):
                    mm.L.mnb_debug_set_infl_skip(mm._ctx, on)
                    I = InflationLayer(mm).waveCostInflation(le)
                    res[on] = (I["kernel_ms"], I["recomputes"], I["dist"])
                mm.L.mnb_debug_set_infl_skip(mm._ctx, 1)
                out["inflation_clean_candidate_skip"] = {
                    "kernel_ms": res[1][0], "without_skip_kernel_ms": res[0][0], "recomputes": int(res[1][1]), "without_skip_recomputes": int(res[0][1]),
                    "identical": bool((res[1][2].view(np.uint32) == res[0][2].view(np.uint32)).all())}
            # the layer walk: round 1's thread-local form (mode 0), the prefetching walk (2) and the default (5: compact seen-set)
            res = {}
            try:
                for mode in (0, 2, 5):
                    mm.L.mnb_debug_set_layers_smem(mm._ctx, mode)
                    for rep in range(2):
                        res[mode] = mm.computeLayers()
                same = all(bool((res[m][k].view(np.uint32) == res[0][k].view(np.uint32)).all()) for m in (2, 5)
                           for k in ("height_diff", "roughness", "steepness", "ridge", "combined"))
                out["layers_prefetching_walk_vs_round1_walk"] = {
                    "kernel_ms": res[5]["kernel_ms"], "prefetching_walk_32bit_seen_set_kernel_ms": res[2]["kernel_ms"], "round1_walk_kernel_ms": res[0]["kernel_ms"],
                    "hbm_frac": 837 * V / (res[5]["kernel_ms"] * 1e-3) / 1e9 / hbm0, "identical": same}
            finally:
                mm.L.mnb_debug_set_layers_smem(mm._ctx, 5)
            return out

        leg("dijkstra_full_field", leg_dijkstra)
        leg("fused_layers", leg_layers)
        leg("inflation", leg_inflation)
        if not args.no_config3:
            leg("config3_plan", leg_config3)
        leg("dynamic_obstacle_update", leg_dynamic_update)
        leg("make_plan_corner_to_corner", leg_make_plan)
        leg("obstacle_raycast", leg_obstacle_raycast)
        leg("optin_variants", leg_optin_variants)
        if n >= args.submesh_from and not args.no_cpu_baseline:
            leg("submesh_1m_parity", leg_submesh_parity)
        shared.clear()

    exit_code = 0
    if rank == 0:
        hbm, which = peaks()
        k_ms = float(np.mean(kernel_ms))
        achieved = CVP_BYTES_PER_VERTEX * settled / (k_ms * 1e-3) / 1e9
        traffic = ncu_traffic(f"cvp_full_field_terrain_{n}x{n}")
        config = {"workload": f"cvp_full_field_terrain_{n}x{n}", "vertices": V, "faces": mm.F, "edges": E,
                  "plans_per_step_per_gpu": 1, "sharding": "one goal per GPU (distinct goals within 2% of the map centre: same wave depth on every rank), potentials all-gathered (NCCL)" if world > 1 else "single GPU",
                  "l2": "256 MB buffer rewritten between timed iterations; working set (>500 MB) exceeds L2",
                  "parity": None, "config3": (other or {}).get("config3_plan"), "batched": batched}
        line = {
            "metric": METRIC, "value": value, "unit": "vertices/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 update / f32 store", "data": "synthetic",
            "config": config,
            "e2e": {"value": e2e_value, "unit": "vertices/s", "h2d_bytes_per_step": int(4 * V + 4 * E),
                    "d2h_bytes_per_step": int(16 * V), "steps": e2e_steps},
            "gpu_launches": int(args.steps * st["kernel_launches"]),
            "roofline": {"bound": "hbm", "kernel": "k_cvp_grid", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                         "frac": achieved / hbm, "traffic": traffic["bytes"] if isinstance(traffic, dict) else traffic,
                         "traffic_source": traffic.get("source") if isinstance(traffic, dict) else None, "peak_source": which,
                         "kernel_ms": k_ms, "rounds": int(st["rounds"]), "recomputes_per_vertex": st["recomputes"] / V,
                         "deep_cascade_labels": int(st.get("deep_labels", 0)),
                         "batched_plans_per_s": batched.get("plans_per_s") if batched else None,
                         "batched_hbm_frac": batched.get("roofline_hbm_frac_rank0") if batched else None,
                         "note": "single wavefront is dependency-latency bound (SURVEY.md H3)"},
            "clocks": clocks,
        }
        if batched:
            line["batched"] = batched
        if other:
            line["other_kernels"] = other
        if not args.no_cpu_baseline:
            from oracle import oracle as O
            flags = O.use_native_build()             # -O3 -march=native on this host (BASELINE.md section 2)
            om = O.OracleMesh(pos, faces)            # same mesh, same goal as the timed plans
            bed = om.edge_distances(); bvc = np.zeros(om.V, np.float32)
            # parity of the TIMED plan: the oracle's plan on the same input in canonical tie order
            ref = om.cvp(bed, bvc, sf, sp)
            config["parity"] = parity_block(h_timed["dist"], h_timed["pred"], ref, h_timed["cut"])
            config["parity"]["deep_cascade_labels"] = int(st.get("deep_labels", 0))
            tot_s, tot_v, reps = 0.0, 0, 0
            while tot_s < 6.0 and reps < 10:
                r = om.cvp(bed, bvc, sf, sp, canonical_ties=False)
                tot_s += r["seconds"]; tot_v += int(np.isfinite(r["dist"]).sum()); reps += 1
            line["cpu_baseline"] = {"value": tot_v / tot_s, "unit": "vertices/s", "cores": 1, "kind": "port", "flags": flags,
                                    "sample": f"{reps} full-field CVP plans on the same {n}x{n} terrain (heap loop only); "
                                              "the reference's loop is single-threaded per plan"}
            bad = [k for k, pbk in (("headline", config["parity"]), ("config3", (config["config3"] or {}).get("parity")),
                                    ("batched", (batched or {}).get("parity_sampled"))) if pbk is not None and not pbk.get("ok", True)]
            if bad:
                line["parity_failed"] = bad
                exit_code = 3
        print(json.dumps(line))
    mm.close()
    if world > 1:
        dist.destroy_process_group()
    if exit_code:
        sys.exit(exit_code)       # the line above is printed either way; a parity failure must not pass silently


if __name__ == "__main__":
    main()
