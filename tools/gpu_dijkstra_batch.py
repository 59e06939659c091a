"""Batched full-field Dijkstra (mnb_dijkstra_batch) on the 1M-vertex terrain with the config-4 goals, against a loop of
single full-field plans (mnb_dijkstra) over the same goals and, for context, the CVP batch (mnb_cvp_batch).

    python tools/gpu_dijkstra_batch.py [--size 1000] [--goals 1024] [--loop-goals 1024] [--out profiles/dijkstra_batch_b200.json]

Costs 0, edge_cost_factor 0, cost_limit 1.  Every leg is warmed up once, then timed: the host clock around the call (each
call ends in a stream synchronise) and the library's CUDA-event kernel time (mnb_get_stats).  The working set (1M-vertex
tables + the [goals][V] rows) is far larger than the L2.  8 sampled rows of the batch are compared with the oracle (distances
bit for bit, predecessors exactly).  The card's name and power limit are read in the same run (nvidia-smi --query-gpu)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1000, help="grid side: size^2 vertices")
    ap.add_argument("--goals", type=int, default=1024)
    ap.add_argument("--loop-goals", type=int, default=1024, help="goals of the single-plan loop (the first ones of the batch)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "dijkstra_batch_b200.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    from mesh_navigation_b200 import synth
    from mesh_navigation_b200.api import MeshMap
    from oracle import oracle as O

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    n = args.size
    pos, faces = synth.grid_mesh(n, n, terrain=True, seed=42)
    mm = MeshMap(pos, faces, device=0)
    V = mm.V
    vc = np.zeros(V, np.float32)
    w = mm.computeEdgeWeights(vc, 0.0)
    goals = synth.batch_goal_vertices(V, args.goals, seed=1234).astype(np.uint32)
    G = goals.size
    gi, gj = np.minimum(goals % n, n - 2), np.minimum(goals // n, n - 2)
    sfs = (2 * (gj * (n - 1) + gi)).astype(np.uint32)
    sps = pos[faces[sfs]].mean(1).astype(np.float32)
    d_dist = torch.empty((G, V), dtype=torch.float32, device="cuda")
    d_pred = torch.empty((G, V), dtype=torch.int32, device="cuda")
    mm.use_device_pointers(True)

    def timed(call, reps):
        call()                                     # warm-up
        wall, kern, st = [], [], None
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call()
            torch.cuda.synchronize()
            wall.append(time.perf_counter() - t0)
            st = mm.stats(); kern.append(st["kernel_ms"])
        return wall, kern, st

    res = {"gpu": gpu, "mesh_vertices": int(V), "goals": int(G), "workload": f"{n}x{n} fBm terrain (seed 42), costs 0, edge_cost_factor 0, "
           "cost_limit 1, goals synth.batch_goal_vertices(V, 1024, seed=1234)", "timing": "host clock around synchronous calls; "
           "kernel_ms = CUDA events inside the library (mnb_get_stats)", "legs": {}}
    for name, call in (("dijkstra_batch_pred", lambda: mm.dijkstra_batch_dev(goals, 1.0, d_dist.data_ptr(), d_pred.data_ptr())),
                       ("dijkstra_batch_nopred", lambda: mm.dijkstra_batch_dev(goals, 1.0, d_dist.data_ptr(), 0)),
                       ("cvp_batch", lambda: mm.cvp_batch_dev(sfs, sps, 1.0, d_dist.data_ptr()))):
        wall, kern, st = timed(call, args.reps)
        res["legs"][name] = {"goals": int(G), "wall_s": wall, "kernel_ms": kern, "plans_per_s": G / min(wall),
                             "rounds_sum": int(st["rounds"]), "relaxations": int(st["recomputes"]), "settled": int(st["settled"])}
        print(name, json.dumps(res["legs"][name]), flush=True)
    # the single-plan loop: whole-GPU cooperative plans, one after the other, into one row
    L = min(args.loop_goals, G)
    loop = lambda: [mm.dijkstra_dev(int(goals[k]), -1, 1.0, 0.3, d_dist.data_ptr(), d_pred.data_ptr()) for k in range(L)]
    mm.dijkstra_dev(int(goals[0]), -1, 1.0, 0.3, d_dist.data_ptr(), d_pred.data_ptr())
    torch.cuda.synchronize()
    t0 = time.perf_counter(); loop(); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    res["legs"]["dijkstra_single_loop"] = {"goals": int(L), "wall_s": [dt], "plans_per_s": L / dt}
    print("dijkstra_single_loop", json.dumps(res["legs"]["dijkstra_single_loop"]), flush=True)
    res["batch_over_loop_plans_per_s"] = res["legs"]["dijkstra_batch_pred"]["plans_per_s"] / res["legs"]["dijkstra_single_loop"]["plans_per_s"]
    res["batch_nopred_over_loop_plans_per_s"] = res["legs"]["dijkstra_batch_nopred"]["plans_per_s"] / res["legs"]["dijkstra_single_loop"]["plans_per_s"]
    # parity: 8 sampled rows of the batch with predecessors against the oracle
    mm.dijkstra_batch_dev(goals, 1.0, d_dist.data_ptr(), d_pred.data_ptr())
    torch.cuda.synchronize()
    om = O.OracleMesh(pos, faces)
    samp = np.unique(np.linspace(0, G - 1, 8).astype(np.int64))
    nmis = 0
    for k in samp:
        ref = om.dijkstra(w, vc, int(goals[k]))
        got_d = d_dist[int(k)].cpu().numpy(); got_p = d_pred[int(k)].cpu().numpy().view(np.uint32)
        nmis += int((got_d.view(np.uint32) != ref["dist"].view(np.uint32)).sum()) + int((got_p != ref["pred"]).sum())
    res["parity_sampled"] = {"rows": [int(k) for k in samp], "n_mismatch": nmis, "ok": nmis == 0}
    mm.use_device_pointers(False)
    mm.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "batch_over_loop_plans_per_s", "batch_nopred_over_loop_plans_per_s", "parity_sampled")}))


if __name__ == "__main__":
    main()
