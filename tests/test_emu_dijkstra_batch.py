"""tests/test_gpu_dijkstra_batch.py replayed on the CPU interpreter of the kernels (tests/emu, see test_emu_kernels.py): the
batched Dijkstra kernel, its host code and the sharded entry points against the oracle without a GPU, once in the normal
schedule and once with randomised warp order (MNB_EMU_SHUFFLE), which turns a missing barrier into a failure."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "tests", "emu", "run_suite.py")


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")])
    return os.path.join(ROOT, "tests", "emu", "libmeshnav_emu.so")


@pytest.mark.parametrize("shuffle", [None, "3"])
def test_dijkstra_batch_suite_on_the_cpu_interpreter(emu_lib, shuffle):
    env = dict(os.environ, MNB_EMU_SMS="4")
    if shuffle:
        env["MNB_EMU_SHUFFLE"] = shuffle
    r = subprocess.run([sys.executable, RUNNER, os.path.join(ROOT, "tests", "test_gpu_dijkstra_batch.py"), "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "not large_mesh"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, f"interpreted kernels disagree with the oracle (shuffle {shuffle}):\n{tail}"
    assert " passed" in r.stdout and " failed" not in r.stdout, tail
