"""The index traversal code of the CUDA library (csrc/common.cuh, csrc/knn_search.cuh) compiled for the host and
checked against brute force: exact NN-1 (ungated, gated, seeded, early-exit) and kNN (k = 2, 3, 20, 31, 32) on sheets,
lattices with exact distance ties, duplicates, far-apart clusters, degenerate clouds and points one float either side of
the cell faces.  This checks the LOGIC the kernels run (box search, hierarchical far search, ring termination, pruning
margins, tie rule) without a GPU; the GPU parity tests (-m gpu) check the kernels themselves.  The host build is test
infrastructure: the shipped library has no CPU path.

The near searches are instantiated with the queue caps the kernels use (common.cuh kNnQueueCap, kKnnQueueCap), and with a
cap of 1, which sends every queued range through the overflow path.  The point sets are also moved 1 km, 10 km and
100 km out, where the grid margin (4e-6 |x|) widens and more kNN queries go to the far traversal."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RUNS = [
    [],
    ["far"],             # EVERY query answered by the hierarchical far traversal alone (oriented brick slabs, a third of
                         # them with an arbitrary direction; thin tilted sheets and thick double sheets among the point sets)
    ["cap1"],
    ["offset=1000"],
    ["offset=10000"],
    ["cap1", "offset=100000"],
]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("emul") / "emul_search")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off",
                           "-I" + os.path.join(ROOT, "leica_point_cloud_processing_b200", "csrc"),
                           os.path.join(ROOT, "tests", "host_emul", "emul_search.cpp"), "-o", exe])
    return exe


def test_traversal_matches_brute_force(emul):
    procs = [subprocess.Popen([emul] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for args in RUNS]   # independent processes: the six runs take the time of one
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for args, p, out in zip(RUNS, procs, outs):
        assert p.returncode == 0, (args, out[-3000:])
        assert "0 failures" in out, (args, out[-3000:])
        assert out.count(": ok") == 10, (args, out[-3000:])
    # far from the origin the near kNN search gives up more queries to the far traversal
    far_knn = [int(o.strip().splitlines()[-1].split("and ")[1].split()[0]) for o in outs]
    assert far_knn[4] > 4 * far_knn[0] and far_knn[5] > far_knn[4], far_knn
