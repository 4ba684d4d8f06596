"""gicpb_group_cloud_difference: Filter::removeFromCloud (reference src/Filter.cpp:176-189) on every GPU of a group.

Each member indexes a window of the subtract cloud's brick planes (its own planes plus a halo that covers the search radius)
and answers the input points of its own planes; the mask rows are assembled from every member's answers.  On a one-GPU box
the members share the device.  Every case compares the group's mask byte for byte, and its kept count, with the
single-context engine and with the oracle."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    from leica_point_cloud_processing_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def _margin(grid_info, sub):
    """GridIndex::build's margin of the subtract grid, in the same float arithmetic."""
    h = np.float32(grid_info["cell_size"])
    fin = sub[np.isfinite(sub).all(1)]
    max_abs = np.float32(max(np.abs(fin.min(0)).max(), np.abs(fin.max(0)).max()))
    return float(h * (np.float32(0.002) + np.float32(5e-7) * np.float32(max(grid_info["dims"])))
                 + np.float32(4e-6) * max_abs)


def _radius_of_halo(planes, h, margin):
    """the largest search radius whose window halo is `planes` brick planes (8 h H >= r + margin + h)"""
    return 8.0 * h * planes - margin - h


class Panel:
    """A 300 k-point panel scan aligned onto its CAD cloud, with FOD blobs; references computed once per threshold."""

    def __init__(self, eng, oracle):
        src, tgt, T_star = synth.make_pair(300_000, 300_000)
        self.input, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, src), n_blobs=20)
        self.sub = tgt
        self.eng, self.oracle = eng, oracle
        self.ref = {}
        self.reference(4e-4)
        gi = eng.grid_info(2)
        self.h = float(gi["cell_size"])
        r3 = _radius_of_halo(3, self.h, _margin(gi, self.sub)) * (1 - 1e-5)
        self.thresholds = [4e-4, 1.2e-2, r3 * r3, 100.0, 0.0, -1.0]  # launch value, code default, H = 3, whole, 0, < 0

    def reference(self, thr):
        if thr not in self.ref:
            m, k = self.eng.cloud_difference(self.input, self.sub, thr)
            om, ok = self.oracle.difference(self.input, self.sub, thr)
            assert k == ok and np.array_equal(m, om), thr
            self.ref[thr] = (m, k)
        return self.ref[thr]


@pytest.fixture(scope="module")
def panel(eng, oracle):
    return Panel(eng, oracle)


def _same(got, want, what):
    m, k = got
    wm, wk = want
    assert m.dtype == np.uint8 and m.shape == wm.shape, what
    bad = np.flatnonzero(m != wm)
    assert bad.size == 0, f"{what}: {bad.size} rows differ, first {bad[:10]}"
    assert k == wk, (what, k, wk)


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_panel_thresholds(panel, n):
    from leica_point_cloud_processing_b200 import EngineGroup
    grp = EngineGroup([0] * n)
    try:
        for thr in panel.thresholds:
            got = grp.cloud_difference(panel.input, panel.sub, thr)
            _same(got, panel.reference(thr), f"N = {n}, thr = {thr}")
            info = [grp.member(r).grid_info(2)["n_indexed"] for r in range(n)]
            print(f"N = {n} thr = {thr:.6g}: kept {got[1]}, subtract points indexed per member {info}")
            if n > 1 and thr == 4e-4:
                assert all(i < len(panel.sub) for i in info), info
                assert sum(info) < 2 * len(panel.sub), info
            if thr == 100.0:
                assert all(i == len(panel.sub) for i in info), info
    finally:
        grp.close()


def _staggered_lattice():
    """40 k points 1 m apart in a plane, every row and column offset by a different fraction of a metre: whatever plane a
    window ends at, some points lie just inside it.  Within 0.5 m of a point there is no other."""
    j, k = np.meshgrid(np.arange(200), np.arange(200), indexing="ij")
    x = j + k / 200.0
    y = k + j / 200.0
    return np.stack([x, y, np.zeros_like(x)], -1).reshape(-1, 3).astype(np.float32) + np.float32(0.37)


@pytest.mark.parametrize("n", [2, 4])
def test_halo_at_its_boundary(eng, oracle, n):
    """Queries displaced from a subtract point by just under (and just over) the search radius, along both long axes; the
    radius is set just below and just above the largest one each halo of H = 1, 2, 3 planes covers.  A halo one plane too
    narrow keeps points near every window edge that one context drops."""
    from leica_point_cloud_processing_b200 import EngineGroup
    sub = _staggered_lattice()
    cell = 0.02
    eng.set_params(cell_size=cell)
    grp = EngineGroup([0] * n)
    try:
        grp.set_params(cell_size=cell)
        eng.cloud_difference(sub[:10], sub, 1e-4)
        gi = eng.grid_info(2)
        assert abs(gi["cell_size"] - cell) < 1e-9
        margin = _margin(gi, sub)
        windows = []
        for planes in (1, 2, 3):
            for side in (1 - 1e-5, 1 + 1e-5):
                r = _radius_of_halo(planes, cell, margin) * side
                assert r < 0.5
                queries = []
                for axis in (0, 1):
                    for f in (1 - 1e-3, 1 + 1e-3):
                        for s in (-1.0, 1.0):
                            q = sub.copy()
                            q[:, axis] += np.float32(s * f * r)
                            queries.append(q)
                q = np.concatenate(queries)
                thr = r * r
                want = eng.cloud_difference(q, sub, thr)
                om, ok = oracle.difference(q, sub, thr)
                assert want[1] == ok and np.array_equal(want[0], om)
                assert 0 < ok < len(q)
                _same(grp.cloud_difference(q, sub, thr), want, f"N = {n}, H = {planes}, r = {r}")
                windows.append(sum(grp.member(i).grid_info(2)["n_indexed"] for i in range(n)))
        print(f"N = {n}: subtract points indexed over all members, per radius: {windows}")
        assert windows == sorted(windows) and windows[-1] > windows[0]
        assert windows[0] < 2 * len(sub)
    finally:
        grp.close()
        eng.set_params(cell_size=0.0)


def _hard_input(panel, rng):
    sub = panel.sub
    lo, hi = sub.min(0), sub.max(0)
    part = panel.input[rng.choice(len(panel.input), 50_001, replace=False)]
    bad = np.array([[np.nan, 0, 0], [0, np.nan, 0], [0, 0, np.nan], [np.inf, 0, 0], [-np.inf, 1, 1], [1, np.inf, 1],
                    [1, 1, -np.inf], [np.nan, np.inf, -np.inf]], np.float32)
    outside = []
    for a in range(3):  # metres beyond every face of the subtract's box, both ends of every axis
        for end, sign in ((lo, -1.0), (hi, 1.0)):
            for d in (0.001, 0.5, 3.0, 40.0):
                p = (lo + hi) / 2
                p = np.repeat(p[None], 3, 0)
                p[:, a] = end[a] + sign * d
                p[1, (a + 1) % 3] = lo[(a + 1) % 3]
                p[2, (a + 2) % 3] = hi[(a + 2) % 3]
                outside.append(p)
    dup = np.repeat(part[:50], 3, 0)  # duplicates of input points, and subtract points themselves (distance 0)
    on_sub = sub[rng.choice(len(sub), 200, replace=False)]
    out = np.concatenate([part, bad, np.concatenate(outside), dup, on_sub, on_sub]).astype(np.float32)
    return out[rng.permutation(len(out))]


def _rows(a, stride):
    r = np.zeros((len(a), stride // 4), np.float32)
    r[:, :3] = a
    if stride >= 16:
        r[:, 3] = 1.0
    return r


@pytest.mark.parametrize("n", [2, 3, 4])
def test_hard_inputs(panel, eng, oracle, n):
    from leica_point_cloud_processing_b200 import EngineGroup
    rng = np.random.default_rng(11 + n)
    inp = _hard_input(panel, rng)
    if len(inp) % n == 0:  # rows that do not split evenly over the members
        inp = inp[:-1]
    grp = EngineGroup([0] * n)
    try:
        for stride in (12, 16, 32):
            i_rows, s_rows = _rows(inp, stride), _rows(panel.sub, {12: 32, 16: 12, 32: 16}[stride])
            for thr in (4e-4, 1.2e-2, 0.0, -1.0):
                want = eng.cloud_difference(inp, panel.sub, thr)
                om, ok = oracle.difference(inp, panel.sub, thr)
                assert want[1] == ok and np.array_equal(want[0], om)
                _same(grp.cloud_difference(i_rows, s_rows, thr), want, f"N = {n}, stride {stride}, thr {thr}")
        for m in (1, n - 1, n + 1):  # fewer input points than members, and a few more
            few = inp[np.isfinite(inp).all(1)][:m]
            _same(grp.cloud_difference(few, panel.sub, 4e-4), eng.cloud_difference(few, panel.sub, 4e-4), f"{m} points")
            _same(grp.cloud_difference(few, panel.sub, 4e-4), oracle.difference(few, panel.sub, 4e-4), f"{m} points")
    finally:
        grp.close()


@pytest.mark.parametrize("n", [2, 4])
def test_degenerate_split_indexes_everything(panel, eng, oracle, n):
    """a subtract cloud of 1 000 points cannot be split by planes (fewer than 1024 N): every member indexes all of it"""
    from leica_point_cloud_processing_b200 import EngineGroup
    rng = np.random.default_rng(5)
    sub = panel.sub[rng.choice(len(panel.sub), 1000, replace=False)]
    inp = _hard_input(panel, rng)
    grp = EngineGroup([0] * n)
    try:
        for thr in (4e-4, 1.2e-2, 0.0, -1.0):
            want = eng.cloud_difference(inp, sub, thr)
            om, ok = oracle.difference(inp, sub, thr)
            assert want[1] == ok and np.array_equal(want[0], om)
            _same(grp.cloud_difference(inp, sub, thr), want, f"N = {n}, thr {thr}")
            assert all(grp.member(r).grid_info(2)["n_indexed"] == 1000 for r in range(n))
    finally:
        grp.close()


def test_three_million_points_on_three_members(eng):
    """above the 2 M-item switch of the far-search tiles"""
    from leica_point_cloud_processing_b200 import EngineGroup
    from oracle.oracle import Oracle
    src, tgt, T_star = synth.make_pair(3_000_000, 3_000_000, length=8.0, width=3.0)
    inp, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, src), n_blobs=20, length=8.0, width=3.0)
    want = eng.cloud_difference(inp, tgt, 4e-4)
    om, ok = Oracle(fast=True).difference(inp, tgt, 4e-4)
    assert want[1] == ok and np.array_equal(want[0], om)
    grp = EngineGroup([0, 0, 0])
    try:
        _same(grp.cloud_difference(inp, tgt, 4e-4), want, "3 M")
        info = [grp.member(r).grid_info(2)["n_indexed"] for r in range(3)]
        print("3 M points: subtract points indexed per member", info)
        assert all(i < len(tgt) for i in info)
    finally:
        grp.close()


def test_alignment_state_survives_and_members_stay_whole(panel, eng, oracle):
    from leica_point_cloud_processing_b200 import Engine, EngineGroup
    s, t, _ = synth.make_pair(60_000, 60_000)
    grp = EngineGroup([0, 0])
    try:
        grp.set_params(max_corr_distance=1.0)
        grp.set_clouds(t, s)
        first = grp.align()
        shards = [grp.member(r).shard_info() for r in range(2)]
        _same(grp.cloud_difference(panel.input, panel.sub, 4e-4), panel.reference(4e-4), "between aligns")
        again = grp.align()
        assert again["transform"].tobytes() == first["transform"].tobytes()
        for k in ("outer_iterations", "inner_iterations", "cost_evaluations", "corr_pairs_last"):
            assert again[k] == first[k], k
        assert [grp.member(r).shard_info() for r in range(2)] == shards
        fresh = Engine(0)
        try:
            fresh.difference_set_subtract(panel.sub)
            want = fresh.difference_run(panel.input, 1.2e-2)
            res = fresh.cloud_resolution(2)
        finally:
            fresh.close()
        n = len(panel.sub)
        for r in range(2):
            m = grp.member(r)
            assert m.grid_info(2)["n_indexed"] < n      # the member's window of the subtract cloud
            _same(m.difference_run(panel.input, 1.2e-2), want, f"member {r} alone")
            assert m.grid_info(2)["n_indexed"] == n     # ... indexed whole before it answered alone
            # the same sum over the same points, added in the order of another brick numbering
            assert abs(m.cloud_resolution(2) - res) <= 2 * n * 2.0 ** -53 * res
    finally:
        grp.close()


def _lib_args(a):
    a = np.ascontiguousarray(a, np.float32)
    return a, a.ctypes.data, len(a), a.strides[0]


def test_argument_errors_match_one_context(panel, eng):
    from leica_point_cloud_processing_b200 import EngineGroup
    grp = EngineGroup([0, 0])
    lib = grp.lib
    try:
        inp, iptr, n, ist = _lib_args(panel.input[:5000])
        sub, sptr, ns, sst = _lib_args(panel.sub)
        nan = np.full((2000, 3), np.nan, np.float32)
        mask = np.zeros(n, np.uint8)
        kept = ctypes.c_int64()
        cases = {
            "null mask": (iptr, n, ist, sptr, ns, sst, None),
            "bad input stride": (iptr, n, 13, sptr, ns, sst, mask.ctypes.data),
            "bad subtract stride": (iptr, n, ist, sptr, ns, 8, mask.ctypes.data),
            "empty input": (iptr, 0, ist, sptr, ns, sst, mask.ctypes.data),
            "empty subtract": (iptr, n, ist, sptr, 0, sst, mask.ctypes.data),
            "null input": (None, n, ist, sptr, ns, sst, mask.ctypes.data),
            "no finite subtract point": (iptr, n, ist, nan.ctypes.data, len(nan), 12, mask.ctypes.data),
        }
        for name, (ip, ni, si, sp, nsub, ss, mp) in cases.items():
            rc_one = lib.gicpb_cloud_difference(eng.h, ip, ni, si, sp, nsub, ss, 0, 4e-4, mp, ctypes.byref(kept))
            msg_one = lib.gicpb_last_error(eng.h)
            rc = lib.gicpb_group_cloud_difference(grp.h, ip, ni, si, sp, nsub, ss, 4e-4, mp, ctypes.byref(kept))
            assert rc_one != 0 and rc == rc_one, (name, rc, rc_one)
            assert lib.gicpb_group_last_error(grp.h) == msg_one, name
            with pytest.raises(Exception):
                grp._check(rc)
        # and the group still works
        _same(grp.cloud_difference(panel.input, panel.sub, 4e-4), panel.reference(4e-4), "after the errors")
    finally:
        grp.close()


def test_whole_cloud_uploads_per_member():
    """GICPB_SHARD_UPLOAD=0: every member uploads both clouds whole; same answer"""
    code = f"""
import sys, numpy as np
sys.path.insert(0, {ROOT!r})
from leica_point_cloud_processing_b200 import Engine, EngineGroup, synth
src, tgt, T = synth.make_pair(200_000, 200_000)
inp, _ = synth.add_fod_blobs(synth.apply_rigid(T, src), n_blobs=10)
rows = np.zeros((len(inp), 8), np.float32); rows[:, :3] = inp
grp = EngineGroup([0, 0, 0])
kept = []
for thr in (4e-4, 1.2e-2):
    want = Engine(0).cloud_difference(inp, tgt, thr)
    got = grp.cloud_difference(rows, tgt, thr)
    assert got[1] == want[1] and np.array_equal(got[0], want[0]), thr
    kept.append(got[1])
assert kept[0] > 0
print("same mask, kept", kept)
"""
    run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, GICPB_SHARD_UPLOAD="0"))
    print(run.stdout[-2000:], run.stderr[-2000:])
    assert run.returncode == 0
    assert "same mask" in run.stdout


def test_two_gpus(panel):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from leica_point_cloud_processing_b200 import EngineGroup
    grp = EngineGroup([0, 1])
    try:
        for thr in panel.thresholds:
            _same(grp.cloud_difference(panel.input, panel.sub, thr), panel.reference(thr), f"[0, 1] thr {thr}")
    finally:
        grp.close()


def test_cpp_shim_prints_the_same_with_a_group(tmp_path, cube_pair):
    """the drop-in's removeFromCloud under GICPB_DEVICES=0,0 goes through the group: every RESULT line as without it"""
    from oracle import cloud_io as oio
    pkg = os.path.join(ROOT, "leica_point_cloud_processing_b200")
    exe = str(tmp_path / "test_shim")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_shim.cpp"), "-o", exe, "-L" + pkg, "-lgicp_b200",
                           "-Wl,-rpath," + pkg])
    src, tgt, _ = cube_pair
    src.astype(np.float32).tofile(str(tmp_path / "source.f32"))
    tgt.astype(np.float32).tofile(str(tmp_path / "target.f32"))
    s32 = src.astype(np.float32)
    oio.pcd_write(str(tmp_path / "source.pcd"), [("x", 4, "F", 1), ("y", 4, "F", 1), ("z", 4, "F", 1)],
                  [s32[:, 0], s32[:, 1], s32[:, 2]], "binary_compressed")
    p_src, p_tgt, T_star = synth.make_pair(60_000, 60_000)
    fod_aligned, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, p_src), n_blobs=6)
    synth.apply_rigid(np.linalg.inv(T_star), fod_aligned).astype(np.float32).tofile(str(tmp_path / "scan.f32"))
    p_tgt.astype(np.float32).tofile(str(tmp_path / "cad.f32"))
    args = [exe] + [str(tmp_path / f) for f in ("source.f32", "target.f32", "source.pcd", "scan.f32", "cad.f32")]
    outs = {}
    for devices in (None, "0,0"):
        env = {k: v for k, v in os.environ.items() if k not in ("GICPB_DEVICES", "GICPB_DEVICE")}
        if devices:
            env["GICPB_DEVICES"] = devices
        run = subprocess.run(args, capture_output=True, text=True, timeout=600, env=env)
        print(devices, run.stdout[-3000:], run.stderr[-2000:])
        assert run.returncode == 0
        outs[devices] = [l for l in run.stdout.splitlines() if l.startswith("RESULT ")]
    assert outs[None] and outs["0,0"] == outs[None]
