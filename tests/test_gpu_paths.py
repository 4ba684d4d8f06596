"""The paths that every real job runs but that the other parity tests reach only through the final transform, each against
the oracle pass by pass:

A. the seeded correspondence pass (every outer iteration after the first: more probe rings, the previous pass's match as the
   first candidate) over a pose sequence with fresh, stale, out-of-gate and width-changed seeds;
B. the fitness pass seeded with the pairs of the last correspondence pass, and a finite max_range;
C. the search kernels on both sides of the 2 M-item switch of far_tile_for (128-query tiles up to 2,000,000 items, 256 above),
   and a whole 2.3 M-point job (kNN, covariances, both correspondence passes, fitness, normals, resolution) on the 256 tiles;
D. the resident cost kernel in every block shape it takes (512 x 2 below 2 M pairs, 512 x 3 from 2 M on, and the edges of the
   resident / streamed split per block) against the oracle and the per-launch kernel, and its epoch wrap;
E. a member of an EngineGroup used on its own: a plain single-GPU context over the whole source, and the group still right
   afterwards.

A sum of n terms in double differs from any other order of the same sum by at most n * 2^-53 * sum |terms|: a fitness or cost
bound derived from that checks every term, where a hand-picked tolerance could hide a wrong neighbour among millions."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
SWITCH = (1_999_999, 2_000_000, 2_000_001)   # far_tile_for / persistent_variant boundary


def _params(**kw):
    base = dict(max_iterations=100, transformation_epsilon=4e-3, rotation_epsilon=2e-3, max_corr_distance=4e-2,
                k_correspondences=20, gicp_epsilon=1e-3, max_inner_iterations=20, cell_size=0.0, points_per_cell=6.0,
                mahalanobis_fp32=0, use_previous_match=1, cost_moments=0, cost_persistent=1)
    base.update(kw)
    return base


@pytest.fixture(scope="module")
def eng():
    from leica_point_cloud_processing_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def fast_oracle():
    from oracle.oracle import Oracle
    return Oracle(fast=True)


@pytest.fixture(scope="module")
def panel_100k():
    src, tgt, _ = synth.make_pair(100_000, 100_000)
    return src, tgt


def _outliers(n, seed, lo=(-0.2, -1.2, -0.5), hi=(4.2, 1.2, 0.4)):
    """sparse points in the panel's surroundings, mostly centimetres to decimetres off the surface"""
    rng = np.random.default_rng(seed)
    return (np.asarray(lo) + rng.random((n, 3)) * (np.asarray(hi) - np.asarray(lo))).astype(np.float32)


def _assert_pass(name, got, ref, fp32):
    pairs, idx, d2, maha = got
    cnt, oi, od, om = ref
    assert pairs == cnt, (name, pairs, cnt)
    assert (idx != -2).all(), name
    assert np.array_equal(idx, oi), (name, int((idx != oi).sum()))
    hit = oi >= 0
    assert np.array_equal(d2[hit], od[hit]), name
    assert np.isinf(d2[~hit]).all(), name
    # fp32: the kernel rounds its double matrix to float; the oracle's double differs from that double by < 1e-9
    rtol = 2.0 ** -24 if fp32 else 0.0
    assert np.allclose(maha, om, rtol=rtol, atol=1e-9), (name, float(np.abs(maha - om).max()))


# ---- A. seeded correspondence passes -------------------------------------------------------------------------------------
@pytest.mark.parametrize("cloud", ["panel_100k", "cube"])
@pytest.mark.parametrize("gate", [0.04, 1.0])
def test_seeded_correspondences_over_a_pose_sequence(eng, oracle, panel_100k, cube_pair, cloud, gate):
    src, tgt = panel_100k if cloud == "panel_100k" else cube_pair[:2]
    poses = [
        ("first pass", np.zeros(6)),
        ("small step", np.array([0.002, -0.001, 0.0015, 0.001, -0.002, 0.003])),
        ("large jump", np.array([0.05, -0.03, 0.04, 0.06, -0.05, 0.1])),
        ("identity", np.zeros(6)),
        ("seeds out of the gate", np.array([0.9 * gate, 0.3 * gate, 0.0, 0.0, 0.0, 0.0])),
    ]
    for w0 in (0, 1):
        eng.set_params(**_params(max_corr_distance=gate, mahalanobis_fp32=w0))
        eng.set_clouds(tgt, src)
        cov_s, cov_t = eng.covariances(1), eng.covariances(0)
        for step, (name, x) in enumerate(poses):
            # the width changes before "identity": that pass must not take the seeds of the other width
            fp32 = w0 if step < 3 else 1 - w0
            if step == 3:
                eng.set_params(mahalanobis_fp32=fp32)
            T = fast_T(oracle, x)
            got = eng.correspondences(T, seeded=step > 0)
            far = eng.last_far_queries()
            ref = oracle.correspondences(src, tgt, cov_s, cov_t, T, gate)
            print(f"{cloud} gate {gate} fp32 {fp32} {name}: pairs {got[0]} far {far}")
            _assert_pass(f"{cloud} gate {gate} fp32 {fp32} {name}", got, ref, fp32)
    eng.set_params(**_params())


def fast_T(oracle, x):
    return oracle.apply_state(np.asarray(x, np.float64))


# ---- B. seeded fitness -----------------------------------------------------------------------------------------------------
def _fitness_bound(src, tgt, T, ref):
    """n * 2^-53 relative: the mean of <= n positive float32 terms summed in double in any order"""
    return 2.0 * len(src) * U * abs(ref) + 1e-300


def test_seeded_fitness_near_and_far_from_the_pairs(eng, oracle, panel_100k):
    src, tgt = panel_100k
    eng.set_params(**_params(max_corr_distance=1.0))
    eng.set_clouds(tgt, src)
    Ta = fast_T(oracle, [0.01, -0.005, 0.004, 0.01, -0.01, 0.02])
    for name, xb, max_range in (("near", [0.011, -0.004, 0.004, 0.011, -0.009, 0.021], None),
                                ("far", [-0.04, 0.05, -0.03, -0.05, 0.04, -0.09], None),
                                ("near, max_range 1e-4", [0.011, -0.004, 0.004, 0.011, -0.009, 0.021], 1e-4)):
        eng.correspondences(Ta)        # valid pairs: the fitness pass is seeded with them
        Tb = fast_T(oracle, xb)
        if max_range is None:
            fit, ref = eng.fitness(Tb), oracle.fitness(src, tgt, Tb)
        else:
            fit, ref = eng.fitness(Tb, max_range), oracle.fitness(src, tgt, Tb, max_range)
        print(f"fitness {name}: {fit!r} oracle {ref!r} far {eng.last_far_queries()}")
        assert abs(fit - ref) <= _fitness_bound(src, tgt, Tb, ref), (name, fit, ref)
    eng.set_params(**_params())


# ---- C. the 2 M-item switch of the search kernels ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def switch_target():
    return synth.panel_points(200_000, 77)


def _queries(n, seed, far=True):
    """n finite queries: on and off the panel, and (far=True) far outside its bounding box"""
    rng = np.random.default_rng(seed)
    n_far, n_off = (n // 100 if far else 0), n // 10
    on = synth.panel_points(n - n_far - n_off, seed, noise_sigma=2e-3)
    off = _outliers(n_off, seed + 1)
    distant = ((rng.random((n_far, 3)) - 0.5) * 60.0).astype(np.float32)
    q = np.concatenate([on, off, distant])
    return q[rng.permutation(n)]


@pytest.mark.parametrize("n", SWITCH)
def test_nn1_and_fitness_at_the_far_tile_switch(eng, fast_oracle, switch_target, n):
    tgt = switch_target
    eng.set_params(**_params())
    eng.set_target(tgt)
    q = _queries(n, 100 + n % 7)
    T = fast_oracle.apply_state(np.array([0.003, -0.002, 0.001, 0.002, 0.001, -0.004]))
    idx, d2 = eng.nn1(q, T=T)
    far = eng.last_far_queries()
    print(f"nn1 n={n}: far {far}")
    assert far > 0
    oi, od = fast_oracle.nn1(tgt, fast_oracle.transform(T, q))
    assert np.array_equal(idx, oi) and np.array_equal(d2, od)
    # fitness: a source of n finite points (n items), decimetres off the panel at most
    q = _queries(n, 200 + n % 7, far=False)
    eng.set_source(q)
    assert eng.grid_info(1)["n_indexed"] == n
    fit = eng.fitness(T)
    far = eng.last_far_queries()
    ref = fast_oracle.fitness(q, tgt, T)
    print(f"fitness n={n}: {fit!r} oracle {ref!r} far {far}")
    assert far > 0
    assert abs(fit - ref) <= _fitness_bound(q, tgt, T, ref)


def test_whole_job_above_the_switch(eng, fast_oracle):
    """one job of 2,300,001 finite points per cloud (1 % of them sparse outliers): every search runs the 256-query tiles"""
    from _cov_util import normal_error_bound, raw_covariances, regularised_from_svd
    n = 2_300_001
    n_out = n // 100
    tgt = np.concatenate([synth.panel_points(n - n_out, 31), _outliers(n_out, 32)])
    src = np.concatenate([synth.panel_points(n - n_out, 33, noise_sigma=1e-3), _outliers(n_out, 34)])
    gate = 1.0
    eng.set_params(**_params(max_corr_distance=gate))
    eng.set_clouds(tgt, src)
    assert eng.grid_info(0)["n_indexed"] == n and eng.grid_info(1)["n_indexed"] == n
    t0 = time.time()

    idx, d2 = eng.knn(0)
    far = eng.last_far_queries()
    print(f"knn-20 n={n}: far {far}")
    assert far > 0
    oi, od = fast_oracle.knn(tgt, 20)
    assert np.array_equal(idx, oi) and np.array_equal(d2, od)

    cov_t = eng.covariances(0)
    np_ref, sv = regularised_from_svd(raw_covariances(tgt, oi), 1e-3)
    bound = normal_error_bound(sv)
    err = np.abs(cov_t - np_ref).max(axis=(1, 2))
    assert (err <= 2.0 * bound).all(), float((err / bound).max())
    ref_cov = fast_oracle.covariances(tgt)
    assert (np.abs(cov_t - ref_cov).max(axis=(1, 2)) <= 2.0 * bound).all()
    del oi, od, np_ref, sv, ref_cov
    cov_s = eng.covariances(1)

    for mode, x in ((0, [0.004, -0.003, 0.002, 0.002, -0.001, 0.003]), (1, [0.005, -0.002, 0.002, 0.003, -0.002, 0.004])):
        T = fast_oracle.apply_state(np.array(x))
        got = eng.correspondences(T, seeded=mode == 1)
        far = eng.last_far_queries()
        print(f"correspondences {'seeded' if mode else 'first'} n={n}: pairs {got[0]} far {far}")
        assert far > 0
        _assert_pass(f"mode {mode}", got, fast_oracle.correspondences(src, tgt, cov_s, cov_t, T, gate), False)

    Tb = fast_oracle.apply_state(np.array([0.006, -0.002, 0.003, 0.003, -0.002, 0.005]))
    fit = eng.fitness(Tb)
    far = eng.last_far_queries()
    ref = fast_oracle.fitness(src, tgt, Tb)
    print(f"fitness n={n}: {fit!r} oracle {ref!r} far {far}")
    assert far > 0
    assert abs(fit - ref) <= _fitness_bound(src, tgt, Tb, ref)

    mask, kept = eng.normal_validity(0, 0.004)
    omask, okept = fast_oracle.normal_validity(tgt, 0.004)
    print(f"normal validity n={n}: {kept} valid, far {eng.last_far_queries()}")
    assert kept == okept and np.array_equal(mask, omask)

    res = eng.cloud_resolution(0)
    far = eng.last_far_queries()
    ref = fast_oracle.resolution(tgt)
    print(f"resolution n={n}: {res!r} oracle {ref!r} far {far}")
    assert far > 0
    assert abs(res - ref) <= 1e-12 * ref
    print(f"checks of the 2.3 M job: {time.time() - t0:.1f} s")
    eng.set_params(**_params())


# ---- D. the resident cost kernel ---------------------------------------------------------------------------------------------
def _states(k, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((k, 6)) - 0.5) * np.array([0.02, 0.02, 0.02, 0.02, 0.02, 0.04])


def _cost_bounds(orc, src, tgt, idx, maha, x):
    """|f - f_ref| and |g - g_ref| allowed for two orders of the same sums: 2 * n * 2^-53 * sum |terms|, scaled as fdf scales
    the sums (f = s0 / m, g = 2 s / m; the rotation gradient adds 9 entries of dR, each of magnitude <= 2, times the sums)"""
    v = np.nonzero(idx >= 0)[0]
    m = len(v)
    p = src[v].astype(np.float64)
    T = orc.apply_state(x)
    r = orc.transform(T, src[v]).astype(np.float64) - tgt[idx[v]].astype(np.float64)
    Mr = np.einsum("nij,nj->ni", maha[v], r)
    eps_n = 2.0 * m * U
    bf = eps_n * np.abs(np.einsum("ni,ni->n", r, Mr)).sum() / m
    bt = eps_n * 2.0 * np.abs(Mr).sum(axis=0) / m
    br = eps_n * 2.0 * 2.0 * (np.abs(p).T @ np.abs(Mr)).sum() / m
    return bf, np.concatenate([bt, np.full(3, br)])


def _check_cost_sessions(e, orc, cloud, xs, expect_shape):
    """cost_persistent 1 vs 0 vs oracle on the pairs of `cloud` matched with itself (every point one pair)"""
    n = len(cloud)
    out = {}
    for mode in (1, 0):
        e.set_params(cost_persistent=mode)
        out[mode] = e.cost_session(xs)
    f1, g1, info = out[1]
    f0, g0, info0 = out[0]
    print(f"cost session n={n}: {info['threads']} x {info['stages']} ring, {info['blocks']} blocks, "
          f"{info['pairs_per_block']} pairs per block, {info['resident']} resident (cap {info['resident_cap']}), "
          f"{info['launches']} launch(es), epochs {info['epoch_first']}..{info['epoch_last']}")
    assert info["persistent"] == 1 and info["launches"] == 1 and info["n_pairs"] == n
    assert (info["threads"], info["stages"]) == expect_shape
    assert info0["persistent"] == 0 and info0["launches"] == len(xs)
    # one order of the sums per set of pairs and block shape: the same states in another session, in reverse, same bits
    e.set_params(cost_persistent=1)
    fr, gr, _ = e.cost_session(xs[::-1])
    assert np.array_equal(fr[::-1], f1) and np.array_equal(gr[::-1], g1)
    pairs, idx, _, maha = e.correspondences(np.eye(4, dtype=np.float32), seeded=True)   # the same pairs, read back
    assert pairs == n
    valid = np.nonzero(idx >= 0)[0].astype(np.int32)
    worst = 0.0
    for k, x in enumerate(xs):
        fo, go = orc.cost(cloud, cloud, valid, idx[valid], maha, x)
        bf, bg = _cost_bounds(orc, cloud, cloud, idx, maha, x)
        # resident and per-launch kernel: the same terms in two orders; each against the oracle likewise
        for name, f, g in (("resident", f1[k], g1[k]), ("per-launch", f0[k], g0[k])):
            assert abs(f - fo) <= bf, (name, k, f, fo, bf)
            assert (np.abs(g - go) <= bg).all(), (name, k, g, go, bg)
        assert abs(f1[k] - f0[k]) <= bf and (np.abs(g1[k] - g0[k]) <= bg).all(), k
        worst = max(worst, abs(f1[k] - f0[k]) / bf, float((np.abs(g1[k] - g0[k]) / bg).max()))
    print(f"  resident vs per-launch: largest difference {worst:.3g} of the summation bound")
    return info


@pytest.fixture(scope="module")
def big_cloud():
    return synth.panel_points(4_200_001, 55, noise_sigma=5e-4)


@pytest.mark.parametrize("n", SWITCH + (4_200_001,))
def test_resident_cost_kernel_shapes(eng, fast_oracle, big_cloud, n):
    cloud = big_cloud[:n]
    eng.set_params(**_params(max_corr_distance=0.01))
    eng.set_clouds(cloud, cloud)
    xs = _states(6, n % 1000)
    for fp32 in (0, 1):
        eng.set_params(mahalanobis_fp32=fp32, cost_persistent=1)
        pairs, _, _, _ = eng.correspondences(np.eye(4, dtype=np.float32))
        assert pairs == n
        _check_cost_sessions(eng, fast_oracle, cloud, xs, (512, 3) if n >= 2_000_000 else (512, 2))
    eng.set_params(**_params())


_EDGES = r"""
import sys
import numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, {tests!r})
from leica_point_cloud_processing_b200 import Engine, synth
from oracle.oracle import Oracle
from test_gpu_paths import _check_cost_sessions, _states

orc = Oracle(fast=True)
e = Engine(0)
pool = synth.panel_points(600_000, 66, noise_sigma=5e-4)


def per_block(n, blocks):
    return (-(-n // blocks) + 15) & ~15


for fp32 in (0, 1):
    e.set_params(max_corr_distance=0.01, points_per_cell=6.0, mahalanobis_fp32=fp32, cost_persistent=1)
    probe = pool[:20_000]
    e.set_clouds(probe, probe)
    e.correspondences(np.eye(4, dtype=np.float32))
    _, _, info = e.cost_session(_states(1, 0))
    B, C = info["blocks"], info["resident_cap"]
    assert (info["threads"], info["stages"]) == (512, 3) and C % 16 == 0 and C > 0, info
    # (pairs per block, pairs of the last block): streamed pairs of the last block 0 / 1 / 511 / 512 / 513, and an odd last
    # block below the resident cap (its bulk copy of 24-byte rows is rounded up to 16 bytes)
    cases = [(C, C - 1), (C, C // 2 + 1), (C + 16, C + 1), (C + 512, C + 511), (C + 512, C + 512), (C + 528, C + 513)]
    for per, last in cases:
        n = (B - 1) * per + last
        assert per_block(n, B) == per and n <= len(pool), (per, last, n)
        cloud = pool[:n]
        e.set_params(cost_persistent=1)
        e.set_clouds(cloud, cloud)
        assert e.correspondences(np.eye(4, dtype=np.float32))[0] == n
        info = _check_cost_sessions(e, orc, cloud, _states(5, n), (512, 3))
        assert info["pairs_per_block"] == per and info["resident"] == min(per, C)
        print(f"fp32 {{fp32}} n {{n}}: streamed per block {{per - min(per, C)}}, last block {{last}} pairs "
              f"({{last - min(last, C)}} streamed)")
e.close()
print("edges ok")
"""


def test_resident_cost_kernel_block_edges():
    """GICPB_COST_VARIANT=3 (512 x 3 at any size; read once per process) at small pair counts chosen from the reported
    resident cap, so that blocks stream 0, 1, 511, 512 and 513 pairs past what they park"""
    code = _EDGES.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, GICPB_COST_VARIANT="3"))
    print(run.stdout[-4000:], run.stderr[-4000:])
    assert run.returncode == 0 and "edges ok" in run.stdout


def test_cost_epochs_alternate_across_the_wrap(oracle, cube_pair):
    """The resident kernel of one session reads the command slot of its epoch's parity; consecutive sessions must alternate
    slots, also where the 12-bit epoch wraps, so that one launch's EXIT is never overwritten by the next launch's command."""
    from leica_point_cloud_processing_b200 import Engine
    src, tgt, _ = cube_pair
    e = Engine(0)
    try:
        e.set_params(**_params(max_corr_distance=5.0))
        e.set_clouds(tgt, src)
        pairs, idx, _, maha = e.correspondences(np.eye(4, dtype=np.float32))
        xs = _states(4, 9)
        ref = [e.cost_session(x[None])[:2] for x in xs]    # resident kernel: every later session must give these bits
        epochs = []
        for k in range(4100):
            f, g, info = e.cost_session(xs[k % 4][None])
            assert info["launches"] == 1 and info["epoch_first"] == info["epoch_last"]
            epochs.append(info["epoch_first"])
            assert f[0] == ref[k % 4][0][0] and np.array_equal(g[0], ref[k % 4][1][0]), k
        ep = np.array(epochs)
        wraps = np.nonzero(np.diff(ep) < 0)[0]
        print(f"epochs {ep[:3]} ... {ep[wraps[0] - 1:wraps[0] + 3] if len(wraps) else ep[-3:]}; wraps at sessions {wraps}")
        assert len(wraps) >= 1 and ep.min() >= 1 and ep.max() < 4096
        assert ((ep[1:] - ep[:-1]) % 2 != 0).all()          # parity alternates, across the wrap too
        valid = np.nonzero(idx >= 0)[0].astype(np.int32)
        for x, (f, g) in zip(xs, ref):
            fo, go = oracle.cost(src, tgt, valid, idx[valid], maha, x)
            bf, bg = _cost_bounds(oracle, src, tgt, idx, maha, x)
            assert abs(f[0] - fo) <= bf and (np.abs(g[0] - go) <= bg).all()
    finally:
        e.close()


# ---- E. group members on their own -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_group_member_alone_is_a_whole_context(eng, oracle, devices):
    from leica_point_cloud_processing_b200 import EngineGroup
    from oracle.oracle import default_params
    src, tgt, _ = synth.make_pair(60_000, 60_000)
    gate = 1.0
    prm = _params(max_corr_distance=gate)
    ref = oracle.align(src, tgt, default_params(max_corr_distance=gate))
    diag = float(np.linalg.norm(tgt.max(0) - tgt.min(0)))

    def close_to_oracle(res, name):
        assert res["converged"] == 1, name
        assert synth.rotation_error_rad(res["transform"], ref["T"]) <= 1e-4, name
        assert synth.translation_error(res["transform"], ref["T"]) <= 1e-5 * diag, name
        assert res["outer_iterations"] == ref["outer_iterations"], name

    eng.set_params(**prm)
    eng.set_clouds(tgt, src)
    one = eng.align()
    T = one["transform"]
    e_pass = eng.correspondences(T)
    e_cov_s, e_cov_t = eng.covariances(1), eng.covariances(0)
    o_pass = oracle.correspondences(src, tgt, e_cov_s, e_cov_t, T, gate)
    o_fit = oracle.fitness(src, tgt, T)

    grp = EngineGroup(devices)
    try:
        grp.set_params(**prm)
        grp.set_clouds(tgt, src)
        first = grp.align()
        close_to_oracle(first, "group")
        for r in range(grp.size):
            m = grp.member(r)
            got = m.correspondences(T)
            print(f"member {r} of {grp.size}: {int((got[1] == -2).sum())} source points outside its pass, "
                  f"{got[0]} pairs (engine {e_pass[0]})")
            _assert_pass(f"member {r}", got, o_pass, False)
            assert np.array_equal(got[1], e_pass[1]) and np.array_equal(got[2], e_pass[2])
            cov = m.covariances(1)
            assert not np.isnan(cov).any(axis=(1, 2)).any()
            assert np.array_equal(cov, e_cov_s)
            fit = m.fitness(T)
            assert abs(fit - o_fit) <= 1e-9 * o_fit, (r, fit, o_fit)
            res = m.align()
            close_to_oracle(res, f"member {r} align")
            assert res["outer_iterations"] == one["outer_iterations"]
            assert np.allclose(res["transform"], one["transform"], atol=1e-6)
        again = grp.align()
        close_to_oracle(again, "group after its members were used alone")
        assert np.allclose(again["transform"], first["transform"], atol=1e-6)
        info = [grp.member(r).shard_info() for r in range(grp.size)]
        assert sum(hi - lo for lo, hi, _, _ in info) == len(src), info
    finally:
        grp.close()
        eng.set_params(**_params())
