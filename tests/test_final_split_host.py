"""The batch verifier's split tail on the CPU (nvcc host compile of the engine headers, sequential reference executors):
the product of 16 per-window Miller values on [256^w]-scaled G2 lines, after one final exponentiation, is the GT element of the
single check on the Horner-combined points -- for true relations (with identity windows and the [s]G fold of window 0) and for
perturbed ones (one-pair windows in either slot).  tools/hosttest/final_split_host.cu."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "kzg_rs_b200", "csrc")
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not found")


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("split") / "final_split_host")
    subprocess.check_call(["nvcc", "-std=c++17", "-O1", "-x", "cu", "-I", CSRC, os.path.join(ROOT, "tools", "hosttest", "final_split_host.cu"),
                           "-o", out], stderr=subprocess.DEVNULL)
    return out


@pytest.mark.parametrize("seed", [1, 0x5eed])
def test_split_tail_equals_combined_check(exe, seed):
    res = subprocess.run([exe, "split", str(seed)], capture_output=True, text=True, timeout=1800)
    assert res.returncode == 0, res.stdout + res.stderr
    cases = {}
    for line in res.stdout.split("\n"):
        if line.startswith("case "):
            f = line.split()
            cases[f[1]] = (int(f[3]), int(f[5]), int(f[7]))
    assert cases == {"true": (1, 1, 1), "true_dense": (1, 1, 1), "false_single_pair": (0, 0, 1), "false_b_identity": (0, 0, 1)}, res.stdout
