"""The CUDA kernels' LOGIC on the CPU (no GPU needed): mesh_navigation_b200/csrc/*.cu{,h} is compiled unchanged by g++
against the interpreter in tests/emu/ (fibers = CUDA threads, lock-step warps, one process per CTA for cooperative
launches) and the whole `-m gpu` parity suite is replayed on it through the C ABI.

What this does and does not prove: control flow, indexing, the band engine's round logic, sub-warp shuffles, stage /
sweep bookkeeping and every host-side entry point are exercised bit-for-bit against the oracle; timing, occupancy and
memory-ordering (fences) are not modelled -- `-m gpu` on a B200 remains the parity gate.  The interpreter is test
infrastructure: it is never loaded by the mesh_navigation_b200 package (tests/test_abi.py checks that)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "tests", "emu", "run_suite.py")

# (test file, pytest -k expression) groups; the 1M-vertex property test stays GPU-only
PARITY = "test_gpu_parity.py"
GROUPS = [
    (PARITY, "dijkstra or edge_distances or goal_cutoff_small"),
    (PARITY, "cvp_full_field or cvp_seed or cvp_costs"),
    (PARITY, "cvp_cost_weighted or cvp_batch"),
    (PARITY, "inflation or layers or config3"),
    (PARITY, "irregular or disconnected or vector_maps or backtrack or make_plan or locate"),
    (PARITY, "cancel"),
    ("test_gpu_group.py", "sharded_batch"),
    ("test_gpu_raycast.py", "cast_rays or obstacle_layer or obstacle_update or normal_clearance"),
    ("test_gpu_updates.py", "layer_changed or max_combination or on_input_changed or vector_field or repulsive or clean_candidate or shared_memory_variant or high_degree or edge_cases or goal_cutoff_armed or deeply_nested or backstep_deep or seed_pops_after or never_fixed or batch_engine or abi_argument"),
]
# the same tests under a randomised warp schedule (MNB_EMU_SHUFFLE, see tests/emu/cuda_runtime.h): warps are visited in a
# different order on every scheduler pass and preempted at collectives, which turns a missing barrier into a failure
SHUFFLED = [
    ("test_gpu_updates.py", "layer_changed or on_input_changed or vector_field or clean_candidate", "1"),
    (PARITY, "cvp_full_field or dijkstra_bit_exact or inflation_wave or backtrack or locate", "2"),
]


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")])
    return os.path.join(ROOT, "tests", "emu", "libmeshnav_emu.so")


@pytest.mark.parametrize("fname,expr", GROUPS)
def test_gpu_parity_suite_on_the_cpu_interpreter(emu_lib, fname, expr):
    env = dict(os.environ, MNB_EMU_SMS="4")
    r = subprocess.run([sys.executable, RUNNER, os.path.join(ROOT, "tests", fname), "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", f"({expr}) and not large_mesh"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, f"interpreted kernels disagree with the oracle:\n{tail}"
    assert " passed" in r.stdout and " failed" not in r.stdout, tail


@pytest.mark.parametrize("fname,expr,seed", SHUFFLED)
def test_gpu_suite_under_a_randomised_warp_schedule(emu_lib, fname, expr, seed):
    env = dict(os.environ, MNB_EMU_SMS="4", MNB_EMU_SHUFFLE=seed)
    r = subprocess.run([sys.executable, RUNNER, os.path.join(ROOT, "tests", fname), "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", f"({expr}) and not large_mesh"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and " passed" in r.stdout, f"schedule-dependent result (seed {seed}):\n{tail}"


def test_every_parity_test_is_in_a_group():
    """the groups above must cover the whole GPU suite (minus the 1M-vertex test)"""
    import re
    for fname in sorted({f for f, _ in GROUPS}):
        src = open(os.path.join(ROOT, "tests", fname)).read()
        names = re.findall(r"^def (test_\w+)", src, flags=re.M)
        words = [w for f, g in GROUPS if f == fname for w in g.split(" or ")]
        missing = [n for n in names if "large_mesh" not in n and not any(w in n for w in words)]
        assert not missing, f"{fname}: not covered by any interpreter group: {missing}"


def test_cpp_host_mirror_on_the_cpu_interpreter(emu_lib, tmp_path, oracle_mod):
    """tests/cpp/test_planners.cpp (the C++ mirror of the reference's plugin interface, include/meshnav_b200/planners.hpp)
    linked against the interpreted kernels instead of libmeshnav_b200.so"""
    link_dir = tmp_path / "lib"
    link_dir.mkdir()
    os.symlink(emu_lib, link_dir / "libmeshnav_b200.so")
    exe = str(tmp_path / "test_planners")
    orc = os.path.join(ROOT, "oracle")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "test_planners.cpp"),
                           f"-L{link_dir}", "-lmeshnav_b200", f"-L{orc}", "-loracle", f"-Wl,-rpath,{link_dir}", f"-Wl,-rpath,{orc}"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=900, env=dict(os.environ, MNB_EMU_SMS="4"))
    assert out.returncode == 0, out.stdout + out.stderr
    assert "cpp host mirror ok" in out.stdout


def test_bench_orchestration_on_the_cpu_interpreter(emu_lib, tmp_path, oracle_mod):
    """bench.py's B200 arm, every leg, executed end to end on the interpreter at toy sizes (tests/emu/run_bench_on_emu.py):
    the JSON line must carry every key of the result line and no secondary leg may have fallen into its error branch; the arrays
    --dump-outputs writes must be the timed plan's, i.e. the oracle's plan of the same seeded input"""
    import json
    import runpy

    import numpy as np
    dump = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "run_bench_on_emu.py"), "--size", "90", "--batch-size", "50",
                        "--batch-goals", "4", "--batch-steps", "1", "--steps", "1", "--warmup", "1", "--dump-outputs", str(dump)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "e2e", "gpu_launches", "roofline", "clocks", "cpu_baseline", "batched", "other_kernels"):
        assert k in line, k
    assert line["metric"] == "vertex-relaxations/sec" and "workload" in line["config"] and line["gpu_launches"] > 0
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in line["roofline"], k
    assert "error" not in line["batched"], line["batched"]
    for name, leg in line["other_kernels"].items():
        assert "error" not in leg, (name, leg)
    assert line["other_kernels"]["dynamic_obstacle_update"]["incremental_equals_full"] is True
    v = line["other_kernels"]["optin_variants"]
    assert v["layers_prefetching_walk_vs_round1_walk"]["identical"] and v["inflation_clean_candidate_skip"]["identical"]
    # the parity blocks of the driver-run line: timed plan, config-3 plan, sampled batch fields
    assert line["config"]["parity"]["ok"] and line["config"]["parity"]["n_mismatch"] == 0
    assert line["config"]["config3"]["parity"]["ok"] and line["config"]["batched"]["parity_sampled"]["ok"]
    assert "parity_failed" not in line
    got = {k: np.load(dump / f"{k}.npy") for k in ("vertex_index", "dist", "pred", "direction", "cutting_face")}
    assert sum(os.path.getsize(dump / f"{k}.npy") for k in got) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    B = runpy.run_path(os.path.join(ROOT, "bench.py"))
    pos, faces = B["build_workload"](90)
    ref = oracle_mod.OracleMesh(pos, faces)
    ref = ref.cvp(ref.edge_distances(), np.zeros(ref.V, np.float32), *B["goal_for_rank"](pos, faces, 90, 0))
    idx = got["vertex_index"].astype(np.int64)
    assert np.array_equal(idx, np.arange(ref["dist"].size))
    assert (got["dist"].view(np.uint32) == ref["dist"][idx].view(np.uint32)).all()
    assert (got["pred"] == ref["pred"][idx]).all() and (got["cutting_face"] == ref["cutting_face"][idx]).all()
    assert np.array_equal(got["direction"], ref["direction"][idx], equal_nan=True)


def test_smoke_entry_on_the_cpu_interpreter(emu_lib):
    """__graft_entry__.smoke() (the driver's GPU smoke check) with the binding pointed at the interpreted kernels"""
    code = ("import sys; sys.path.insert(0, %r); from mesh_navigation_b200 import _lib; _lib.LIB_PATH = %r; "
            "import __graft_entry__ as g; g.smoke()") % (ROOT, emu_lib)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, MNB_EMU_SMS="4"))
    assert r.returncode == 0 and "smoke ok" in r.stdout, (r.stdout + r.stderr)[-2000:]


def test_interpreter_self_test(tmp_path):
    """the interpreter's warp / block / grid primitives against the semantics the CUDA programming guide documents
    (tests/emu/selftest/selftest.cu): segment shuffles, votes and reductions with exited lanes, 64-bit payloads, block
    barriers with exited threads, a cooperative launch with grid barriers and global atomics across CTA processes"""
    exe = str(tmp_path / "emu_selftest")
    emu = os.path.join(ROOT, "tests", "emu")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-strict-aliasing", "-Wno-unknown-pragmas",
                           "-Wno-attributes", f"-I{emu}", "-x", "c++", os.path.join(emu, "selftest", "selftest.cu"), "-o", exe])
    for env in ({}, {"MNB_EMU_SHUFFLE": "5"}):
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=dict(os.environ, **env))
        assert r.returncode == 0 and "interpreter self-test ok" in r.stdout, r.stdout + r.stderr
