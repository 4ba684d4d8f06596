"""The exact NN-1 passes (csrc/nn_kernels.cu: correspondence_kernel, fitness_kernel, difference_kernel, nn1_kernel and
transform_kernel) at their edges, against the oracle.

Each pass decides by the float d2 of FLANN's order, (dx*dx + dy*dy) + dz*dz, and by PCL's comparison of that float with a
double limit: d2 < gate^2 (GICP pairs), d2 > threshold (getPointCloudDifference keeps the point), d2 <= max_range
(getFitnessScore counts it).  So the decisions are compared bit for bit.

What a case asserts:
  * correspondences(T, seeded): pair count, idx and d2 equal Oracle.correspondences' bit for bit (-2 on non-finite source
    rows, the oracle run on the finite rows of both clouds and its indices mapped back); maha within 1e-9 (exact width)
    or 2^-24 relative (fp32 width); both widths;
  * nn1: idx and d2 equal Oracle.nn1's, gated as the hook gates (d2 < max_dist^2 for max_dist > 0) where the case is
    about the gate;
  * fitness(T[, max_range]), unseeded and seeded: within 2 n 2^-53 |ref|, the bound of two summation orders;
  * cloud_difference: mask and kept count equal Oracle.difference's;
  * cost / cost_session on the pairs of the case: within the summation bounds of _cost_bounds;
  * where a case is built for it, last_far_queries() > 0 (the far instance ran) or == 0.

Cases: A the cube and a 30 k panel pair 0 m to 10 km out (both passes, fitness, cost, difference, transform, and one
align 300 m out); B queries far off a panel 1 km and 10 km out, and queries 100 m to 10 km from a panel at the origin,
so that the oriented slab cuts decide; C exact ties (lattice edge / face / cell midpoints, a seed that ties with a lower
index, copies); D d2 one float either side of the gate, the threshold and max_range, 0 and 1 km out, and a gate of
1e-30; E non-finite rows and non-finite or out-of-range limits; F a 1 M-point pair 1 km out.

CPU part (-m "not gpu"): the fixtures are what they claim (exact lattices, complete tie sets, the boundary d2 values
attained and straddling each limit, the oracle's decisions equal to a numpy restatement of PCL's comparisons).
"""
import contextlib
import time

import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth

OFFSET_DIR = np.array([1.0, -0.5, 0.25])
SP = 2.0 ** -6                      # tie lattice spacing: every coordinate and every d2 is an exact float
U = 2.0 ** -53
FLT_MAX = float(np.finfo(np.float32).max)
E_BADARG, E_NOT_ENOUGH_CORRESPONDENCES = -1, -4
EYE = np.eye(4, dtype=np.float32)


@contextlib.contextmanager
def timed(label):
    t0 = time.perf_counter()
    yield
    print(f"[time] {label}: {time.perf_counter() - t0:.2f} s")


# ---- fixtures ---------------------------------------------------------------------------------------------------------
def shifted(cloud, offset):
    return (cloud.astype(np.float64) + OFFSET_DIR * offset).astype(np.float32)


@pytest.fixture(scope="module")
def panel_pair():
    src, tgt, _ = synth.make_pair(30_000, 30_000)
    return src, tgt


@pytest.fixture(scope="module")
def fast_oracle():
    from oracle.oracle import Oracle
    return Oracle(fast=True)


def rigid(center, angle, t):
    """float32 4x4: a small rotation about `center` (axis (1, 2, 3)) and a translation, as a pose near the clouds"""
    return synth.rigid_about(np.asarray(center, np.float64), (1.0, 2.0, 3.0), angle, t).astype(np.float32)


def lattice(offset, side=8, seed=0):
    """side^3 lattice of spacing 2^-6 moved offset * OFFSET_DIR (multiples of 2^-6 for the offsets used), shuffled so
    that the original index decides the ties"""
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3) * SP
    return (g + OFFSET_DIR * offset)[np.random.default_rng(seed).permutation(len(g))].astype(np.float32)


def midpoints(offset, side=8):
    """midpoints of the lattice's interior edges (2 equidistant targets), faces (4) and cells (8); with the tie count"""
    rng = np.random.default_rng(1)
    g = np.stack(np.meshgrid(*[np.arange(1, side - 2)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    pts, ties = [], []
    for h, n in (((0.5, 0, 0), 2), ((0, 0.5, 0), 2), ((0, 0, 0.5), 2), ((0.5, 0.5, 0), 4), ((0, 0.5, 0.5), 4),
                 ((0.5, 0, 0.5), 4), ((0.5, 0.5, 0.5), 8)):
        pts.append(g + h)
        ties += [n] * len(g)
    p = np.concatenate(pts) * SP + OFFSET_DIR * offset
    order = rng.permutation(len(p))
    return p[order].astype(np.float32), np.array(ties)[order]


def x_edge_midpoints(tgt, offset):
    """midpoints m = a + (SP/2, 0, 0) of the interior x edges (a, b): (m, index of a, index of b)"""
    key = {tuple(np.round((p.astype(np.float64) - OFFSET_DIR * offset) / SP).astype(int)): i for i, p in enumerate(tgt)}
    m, ia, ib = [], [], []
    for (x, y, z), i in key.items():
        j = key.get((x + 1, y, z))
        if j is not None and 0 < y < 7 and 0 < z < 7:
            m.append(tgt[i].astype(np.float64) + (SP / 2, 0.0, 0.0))
            ia.append(i)
            ib.append(j)
    return np.array(m, np.float32), np.array(ia), np.array(ib)


def with_copies(base, n_pts, copies, seed):
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(base), n_pts, replace=False)
    c = np.concatenate([base] + [base[pick]] * (copies - 1))
    return c[rng.permutation(len(c))].astype(np.float32)


def with_nonfinite(cloud, seed=6, every=17):
    c = np.array(cloud, np.float32)
    rng = np.random.default_rng(seed)
    c[::every, rng.integers(0, 3)] = np.nan
    c[5::every * 3, 1] = np.inf
    c[9::every * 5, 2] = -np.inf
    return c


def _sheet_normal(p):
    """unit radial direction of the panel's base cylinder (synth.panel_points, radius 3) at p"""
    ang = np.arctan2(p[:, 1].astype(np.float64), p[:, 2].astype(np.float64) + 3.0)
    return np.stack([np.zeros_like(ang), np.sin(ang), np.cos(ang)], 1)


def off_surface_queries(offset, n=6000, seed=21):
    """queries 1 cm to 5 m off the panel along its normal (both sides), and beyond its four edges, offset * OFFSET_DIR
    out"""
    rng = np.random.default_rng(seed)
    on = synth.panel_points(n, seed).astype(np.float64)
    dist = np.exp(rng.uniform(np.log(0.01), np.log(5.0), n)) * rng.choice([-1.0, 1.0], n)
    off = on + _sheet_normal(on) * dist[:, None]
    lat = synth.panel_points(n // 3, seed + 1).astype(np.float64)
    lat[:, 0] += rng.choice([-1.0, 1.0], len(lat)) * (4.0 + rng.uniform(0.01, 3.0, len(lat)))
    lat[:, 1] += rng.normal(0, 0.5, len(lat))
    return (np.concatenate([off, lat]) + OFFSET_DIR * offset).astype(np.float32)


def distant_queries(n=4000, seed=22):
    """queries 100 m to 10 km from the origin in every direction"""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return (d * np.exp(rng.uniform(np.log(100.0), np.log(10000.0), n))[:, None]).astype(np.float32)


def outlier_pair(n, offset, seed):
    """a panel pair of n points each with 1 % sparse outliers around it, offset * OFFSET_DIR out"""
    n_out = n // 100
    rng = np.random.default_rng(seed)
    lo, hi = np.array([-0.2, -1.2, -0.5]), np.array([4.2, 1.2, 0.4])
    out_t = lo + rng.random((n_out, 3)) * (hi - lo)
    out_s = lo + rng.random((n_out, 3)) * (hi - lo)
    tgt = np.concatenate([synth.panel_points(n - n_out, seed + 1), out_t])
    src = np.concatenate([synth.panel_points(n - n_out, seed + 2, noise_sigma=1e-3), out_s])
    return shifted(src, offset), shifted(tgt, offset)


# ---- D. the float boundary ---------------------------------------------------------------------------------------------
BOUND_GATES = [0.04, 2.0 ** -4]          # 0.04^2 is not a float, 2^-8 is
BOUND_THRESHOLDS = [0.0016, 2.0 ** -8]
TINY = [0.0, float(np.finfo(np.float32).smallest_subnormal), 1e-23, 1e-22, 1e-19]


def f32d2(q, t):
    """the oracle's (FLANN's) float d2 in its order, elementwise over rows"""
    q, t = np.asarray(q, np.float32), np.asarray(t, np.float32)
    dx, dy, dz = q[..., 0] - t[..., 0], q[..., 1] - t[..., 1], q[..., 2] - t[..., 2]
    return (dx * dx + dy * dy) + dz * dz


def _steps(v, k0, k1):
    """the floats k0 .. k1 steps from the positive float v"""
    return (np.float32(v).view(np.int32) + np.arange(k0, k1, dtype=np.int32)).view(np.float32)


def straddle(t, limit):
    """Queries near target point t whose float d2 to t are the two largest attainable values below `limit` and the two
    smallest at or above it: [(d2, q)] in ascending d2.  q moves from t along x (about sqrt(limit)) and a little along z,
    both found by emulating the float arithmetic (1 km out q - t is a multiple of the coordinate's ulp)."""
    t = np.asarray(t, np.float32)
    xs = _steps(np.float32(np.float64(t[0]) + np.sqrt(limit)), -64, 65)
    ulp = float(np.spacing(np.nextafter(np.float32(limit), np.float32(0))))   # the finer spacing below a power of 2
    zs = np.unique(np.concatenate([
        (np.float64(t[2]) + np.sqrt(np.arange(0, 96) * ulp)).astype(np.float32),
        _steps(t[2], 0, 48) if t[2] > 0 else np.zeros(1, np.float32)]))
    Q = np.empty((len(xs), len(zs), 3), np.float32)
    Q[..., 0] = xs[:, None]
    Q[..., 1] = t[1]
    Q[..., 2] = zs[None, :]
    D = f32d2(Q, t)
    vals = np.unique(D).astype(np.float64)   # compared with the double limit in double, as PCL does
    pick = list(vals[vals < limit][-2:]) + list(vals[vals >= limit][:2])
    out = []
    for v in pick:
        i, j = np.argwhere(D == v)[0]
        out.append((np.float32(v), Q[i, j].copy()))
    return out


def boundary_set(offset):
    """target: 64 points (0, j, 0) shuffled, offset * OFFSET_DIR out (1 m apart: each query's nearest point is
    unambiguous).  Source: per limit of BOUND_GATES^2 and BOUND_THRESHOLDS the four straddling d2 values, the TINY
    offsets along x (d2 0 or subnormal), and 24 fillers 0.01 / 0.3 off.  Returns (tgt, src, intended target index per
    source point, intended d2, {limit: [d2 values]})."""
    base = np.zeros((64, 3))
    base[:, 1] = np.arange(64)
    tgt = (base + OFFSET_DIR * offset)[np.random.default_rng(7).permutation(64)].astype(np.float32)
    src, want_i, want_d2, by_limit = [], [], [], {}
    free = iter(range(64))
    limits = list(dict.fromkeys([g * g for g in BOUND_GATES] + BOUND_THRESHOLDS))   # 0.04^2 == 0.0016 in double
    for L in limits:
        by_limit[L] = []
        j = next(free)
        for v, q in straddle(tgt[j], L):
            src.append(q), want_i.append(j), want_d2.append(v), by_limit[L].append(v)
    for d in TINY:
        j = next(free)
        q = tgt[j].copy()
        q[0] = np.float32(np.float64(q[0]) + d)
        src.append(q), want_i.append(j), want_d2.append(f32d2(q, tgt[j]))
    for k in range(24):
        j = next(free)
        q = tgt[j].astype(np.float64) + ((0.01 if k % 2 else 0.3), 0.0, 0.0)
        q = q.astype(np.float32)
        src.append(q), want_i.append(j), want_d2.append(f32d2(q, tgt[j]))
    return (tgt, np.array(src, np.float32), np.array(want_i), np.array(want_d2, np.float32), by_limit)


# ---- the reference ------------------------------------------------------------------------------------------------------
def finite_rows(c):
    return np.isfinite(c[:, :3]).all(1)


def ref_correspondences(orc, src, tgt, cov_s, cov_t, T, gate):
    """Oracle.correspondences on the finite rows of both clouds, mapped back: -2 / inf / I on non-finite source rows"""
    fs, ft = finite_rows(src), finite_rows(tgt)
    mt = np.flatnonzero(ft)
    cnt, oi, od, om = orc.correspondences(src[fs], tgt[ft], cov_s[fs], cov_t[ft], T, gate)
    idx = np.full(len(src), -2, np.int32)
    idx[fs] = np.where(oi >= 0, mt[np.maximum(oi, 0)], -1)
    d2 = np.full(len(src), np.inf, np.float32)
    d2[fs] = od
    maha = np.tile(np.eye(3), (len(src), 1, 1))
    maha[fs] = om
    return cnt, idx, d2, maha


def ref_nn1(orc, tgt, q, max_dist=0.0):
    """Oracle.nn1 on the finite target rows, gated as gicpb_nn1 gates: d2 < max_dist^2 when max_dist > 0"""
    ft = finite_rows(tgt)
    oi, od = orc.nn1(tgt[ft], q)
    idx = np.where(oi >= 0, np.flatnonzero(ft)[np.maximum(oi, 0)], -1).astype(np.int32)
    if max_dist > 0:
        out = ~(od.astype(np.float64) < max_dist * max_dist)
        idx[out] = -1
        od = np.where(out, np.float32(np.inf), od)
    return idx, od


def reset(engine, **kw):
    base = dict(max_iterations=100, transformation_epsilon=4e-3, rotation_epsilon=2e-3, max_corr_distance=4e-2,
                k_correspondences=20, gicp_epsilon=1e-3, max_inner_iterations=20, cell_size=0.0, points_per_cell=6.0,
                mahalanobis_fp32=0, use_previous_match=1, cost_moments=0, cost_persistent=1)
    base.update(kw)
    engine.set_params(**base)


def assert_pass(name, got, ref, fp32):
    pairs, idx, d2, maha = got
    cnt, oi, od, om = ref
    assert pairs == cnt, (name, pairs, cnt)
    bad = np.flatnonzero(idx != oi)
    assert bad.size == 0, (name, bad.size, bad[:5], idx[bad[:5]], oi[bad[:5]])
    hit = oi >= 0
    assert np.array_equal(d2[hit].view(np.uint32), od[hit].view(np.uint32)), name
    assert np.isinf(d2[~hit]).all(), name
    # fp32: the kernel rounds its double matrix to float; the oracle's double differs from that double by < 1e-9
    rtol = 2.0 ** -24 if fp32 else 0.0
    assert np.allclose(maha, om, rtol=rtol, atol=1e-9), (name, float(np.abs(maha - om).max()))


def check_correspondences(eng, orc, src, tgt, T, gate, seeded, fp32, name, far=None):
    got = eng.correspondences(T, seeded=seeded)
    far_q = eng.last_far_queries()
    ref = ref_correspondences(orc, src, tgt, eng.covariances(1), eng.covariances(0), T, gate)
    print(f"{name} {'seeded' if seeded else 'first'} fp32={fp32}: pairs {got[0]} far {far_q}")
    assert_pass(f"{name} seeded={seeded} fp32={fp32}", got, ref, fp32)
    if far is True:
        assert far_q > 0, f"{name}: the far instance did not run"
    elif far is False:
        assert far_q == 0, f"{name}: far queries ran ({far_q})"
    return got


def check_nn1(eng, orc, tgt, q, name, T=None, max_dist=0.0, far=None):
    idx, d2 = eng.nn1(q, T=T, max_dist=max_dist)
    far_q = eng.last_far_queries()
    qq = q if T is None else orc.transform(T, q)
    ri, rd = ref_nn1(orc, tgt, qq, max_dist)
    bad = np.flatnonzero(idx != ri)
    assert bad.size == 0, (name, bad.size, bad[:5], idx[bad[:5]], ri[bad[:5]], d2[bad[:5]], rd[bad[:5]])
    assert np.array_equal(d2.view(np.uint32), rd.view(np.uint32)), name
    print(f"{name} nn1 max_dist={max_dist}: found {int((idx >= 0).sum())} of {len(q)} far {far_q}")
    if far is True:
        assert far_q > 0, f"{name}: the far instance did not run"
    elif far is False:
        assert far_q == 0, f"{name}: far queries ran ({far_q})"


def check_fitness(eng, orc, src, tgt, T, name, max_range=None, far=None):
    fs, ft = finite_rows(src), finite_rows(tgt)
    if max_range is None:
        fit, ref = eng.fitness(T), orc.fitness(src[fs], tgt[ft], T)
    else:
        fit, ref = eng.fitness(T, max_range), orc.fitness(src[fs], tgt[ft], T, max_range)
    far_q = eng.last_far_queries()
    bound = 2.0 * int(fs.sum()) * U * abs(ref)
    err = abs(fit - ref)
    print(f"{name} fitness max_range={max_range}: {fit!r} oracle {ref!r} far {far_q} "
          f"err/bound {err / bound if bound else 0.0:.3g}")
    assert err <= bound, (name, fit, ref, bound)
    if far is True:
        assert far_q > 0, f"{name}: the far instance did not run"
    return fit


def check_difference(eng, orc, inp, sub, thr, name):
    mask, kept = eng.cloud_difference(inp, sub, thr)
    om, ok = orc.difference(inp, sub[finite_rows(sub)], thr)
    print(f"{name} difference thr={thr!r}: kept {kept} (oracle {ok}) of {len(inp)}, far {eng.last_far_queries()}")
    bad = np.flatnonzero(mask != om)
    assert bad.size == 0 and kept == ok, (name, thr, kept, ok, bad[:5])


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


def cost_states(k, seed):
    """pose increments: centimetres of translation, 1e-5 rad of rotation (about the origin: ~0.1 m at 10 km)"""
    rng = np.random.default_rng(seed)
    return (rng.random((k, 6)) - 0.5) * np.array([0.02, 0.02, 0.02, 2e-5, 2e-5, 2e-5])


def check_cost(eng, orc, src, tgt, got, name, k=3):
    """cost and cost_session (resident kernel) at k states on the pairs of the last correspondence pass"""
    pairs, idx, _, maha = got
    if pairs == 0:
        return
    valid = np.flatnonzero(idx >= 0).astype(np.int32)
    xs = cost_states(k, pairs % 997)
    fs, gs, _ = eng.cost_session(xs)
    worst = 0.0
    for j, x in enumerate(xs):
        f, g = eng.cost(x)
        fo, go = orc.cost(src, tgt, valid, idx[valid], maha, x)
        bf, bg = _cost_bounds(orc, src, tgt, idx, maha, x)
        for which, ff, gg in (("cost", f, g), ("session", fs[j], gs[j])):
            assert abs(ff - fo) <= bf, (name, which, j, ff, fo, bf)
            assert (np.abs(gg - go) <= bg).all(), (name, which, j, gg, go, bg)
            worst = max(worst, abs(ff - fo) / bf, float((np.abs(gg - go) / bg).max()))
    print(f"{name} cost on {pairs} pairs: largest error {worst:.3g} of the summation bound")


# ---- CPU: the fixtures are what they claim ------------------------------------------------------------------------------
def brute(tgt, q):
    """float d2 of every query to every target point, in the oracle's order"""
    return f32d2(q[:, None, :], tgt[None, :, :])


@pytest.mark.parametrize("offset", [0.0, 1024.0])
def test_tie_fixtures_have_2_4_or_8_equidistant_targets(offset):
    tgt = lattice(offset)
    ref = np.round((tgt.astype(np.float64) - OFFSET_DIR * offset) / SP)
    assert np.array_equal(ref * SP + OFFSET_DIR * offset, tgt.astype(np.float64)), "a lattice coordinate is not exact"
    src, ties = midpoints(offset)
    back = (src.astype(np.float64) - OFFSET_DIR * offset) / (SP / 2)
    assert np.array_equal(np.round(back), back), "a midpoint is not exact"
    D = brute(tgt, src)
    m = D.min(1)
    assert np.array_equal((D == m[:, None]).sum(1), ties)
    # the d2 of the 2 / 4 / 8 ties are exact: 1, 2, 3 half spacings squared
    assert np.array_equal(m.astype(np.float64), np.log2(ties) * (SP / 2) ** 2)
    mids, ia, ib = x_edge_midpoints(tgt, offset)
    assert len(mids) > 100 and (ib > ia).any() and (ib < ia).any()
    Dm = brute(tgt, mids)
    assert ((Dm == Dm.min(1)[:, None]).sum(1) == 2).all()
    # shifted 2^-10 towards b, b is the unique nearest
    moved = mids.copy()
    moved[:, 0] = (moved[:, 0].astype(np.float64) + 2.0 ** -10).astype(np.float32)
    assert np.array_equal(moved[:, 0].astype(np.float64), mids[:, 0].astype(np.float64) + 2.0 ** -10)
    Dv = brute(tgt, moved)
    assert np.array_equal(np.argmin(Dv, 1), ib) and ((Dv == Dv.min(1)[:, None]).sum(1) == 1).all()


@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_boundary_values_are_attained_and_straddle(oracle, offset):
    tgt, src, want_i, want_d2, by_limit = boundary_set(offset)
    assert np.array_equal(f32d2(src, tgt[want_i]).view(np.uint32), want_d2.view(np.uint32))
    for L, vals in by_limit.items():
        v = np.array(vals, np.float32)
        assert len(v) == 4 and (v[:2].astype(np.float64) < L).all() and (v[2:].astype(np.float64) >= L).all(), (L, v)
        assert (np.diff(v) > 0).all()
        if offset == 0.0:
            # at the origin the four are consecutive floats: the largest below the limit, the smallest at or above it
            below = np.float32(L)
            if float(below) >= L:
                below = np.nextafter(below, np.float32(0))
            assert v[1] == below and v[2] == np.nextafter(below, np.float32(1)), (L, v)
            assert v[0] == np.nextafter(v[1], np.float32(0)) and v[3] == np.nextafter(v[2], np.float32(1))
    assert float(np.float32(2.0 ** -8)) == 2.0 ** -8 and float(np.float32(0.0016)) != 0.0016
    # every source point's nearest target is the intended one, at the intended d2, and no other target is close
    D = brute(tgt, src)
    assert np.array_equal(np.argmin(D, 1), want_i)
    assert (np.sort(D, 1)[:, 1] > 0.5).all()
    oi, od = oracle.nn1(tgt, src)
    assert np.array_equal(oi, want_i) and np.array_equal(od.view(np.uint32), want_d2.view(np.uint32))
    if offset == 0.0:
        tiny = want_d2[len(by_limit) * 4:len(by_limit) * 4 + len(TINY)]
        assert (tiny[:4] < 1e-43).all() and tiny[4] > 0 and tiny[:2].tolist() == [0.0, 0.0] and (tiny[2:] >= 0).all()


@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_oracle_decisions_restate_pcl(oracle, offset):
    """the oracle's pairs, kept points and fitness on the boundary set equal numpy's restatement of PCL's comparisons of
    the float d2 with a double: d2 < gate^2, d2 > threshold, d2 <= max_range"""
    tgt, src, want_i, want_d2, by_limit = boundary_set(offset)
    d = want_d2.astype(np.float64)
    cov = np.tile(np.eye(3), (64, 1, 1))
    for gate in BOUND_GATES + [1e-30, 0.0, -0.04, np.inf, np.nan]:
        cnt, oi, _, _ = oracle.correspondences(src, tgt, cov[:len(src)], cov, EYE, gate)
        want = d < gate * gate
        assert cnt == int(want.sum()) and np.array_equal(oi >= 0, want), gate
        assert np.array_equal(oi[want], want_i[want])
    assert oracle.correspondences(src, tgt, cov[:len(src)], cov, EYE, 1e-30)[0] == int((want_d2 == 0).sum()) > 0
    for thr in BOUND_THRESHOLDS + [0.0, -1.0, np.inf, 1e300, FLT_MAX, -np.inf, np.nan]:
        mask, kept = oracle.difference(src, tgt, thr)
        want = d > thr
        assert kept == int(want.sum()) and np.array_equal(mask.astype(bool), want), thr
    for mr in sorted(set(by_limit[0.04 * 0.04][2:])) + [0.0, -1.0, np.nan]:
        sel = d <= mr
        ref = d[sel].sum() / sel.sum() if sel.any() else np.finfo(np.float64).max
        got = oracle.fitness(src, tgt, EYE, float(mr))
        assert abs(got - ref) <= 2 * len(d) * U * abs(ref), (mr, got, ref)


# ---- A. far from the origin ---------------------------------------------------------------------------------------------
OFFSETS = [0.0, 300.0, 1000.0, 10000.0]


def _pair(name, cube_pair, panel_pair, offset):
    src, tgt = cube_pair[:2] if name == "cube" else panel_pair
    return shifted(src, offset), shifted(tgt, offset)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("shape", ["cube", "panel"])
def test_far_from_the_origin(engine, oracle, cube_pair, panel_pair, shape, offset):
    src, tgt = _pair(shape, cube_pair, panel_pair, offset)
    c = tgt.astype(np.float64).mean(0)
    T1 = rigid(c, 0.002, (0.003, -0.002, 0.001))
    T2 = rigid(c, 0.0025, (0.0035, -0.0015, 0.001))
    name = f"A {shape} {offset:g} m"
    for gate in (0.04, 1.0):
        for fp32 in (0, 1):
            reset(engine, max_corr_distance=gate, mahalanobis_fp32=fp32)
            engine.set_clouds(tgt, src)
            check_fitness(engine, oracle, src, tgt, T1, f"{name} gate {gate} unseeded")
            check_correspondences(engine, oracle, src, tgt, T1, gate, False, fp32, f"{name} gate {gate}")
            got = check_correspondences(engine, oracle, src, tgt, T2, gate, True, fp32, f"{name} gate {gate}")
            check_fitness(engine, oracle, src, tgt, T2, f"{name} gate {gate} seeded")
            check_fitness(engine, oracle, src, tgt, T2, f"{name} gate {gate} seeded", max_range=1e-4)
            check_cost(engine, oracle, src, tgt, got, f"{name} gate {gate} fp32 {fp32}")
    for thr in (4e-4, 1.2e-2):
        check_difference(engine, oracle, src, tgt, thr, name)
    moved = engine.transform_cloud(T1, src)
    assert np.array_equal(moved.view(np.uint32), oracle.transform(T1, src).view(np.uint32))


@pytest.mark.gpu
def test_align_300_m_out(engine, oracle, panel_pair):
    """every pass is checked bit for bit above: a difference here lies in the loop"""
    from oracle.oracle import default_params
    src, tgt = (shifted(c, 300.0) for c in panel_pair)
    reset(engine, max_corr_distance=1.0)
    engine.set_clouds(tgt, src)
    res = engine.align()
    ref = oracle.align(src, tgt, default_params(max_corr_distance=1.0))
    diag = float(np.linalg.norm(tgt.max(0).astype(np.float64) - tgt.min(0)))
    rot = synth.rotation_error_rad(res["transform"], ref["T"])
    tr = synth.translation_error(res["transform"], ref["T"])
    print(f"A align 300 m: outer {res['outer_iterations']} (oracle {ref['outer_iterations']}) rot {rot:.2e} tr {tr:.2e}")
    assert res["converged"] == ref["converged"] == 1
    assert rot <= 1e-4 and tr <= 1e-5 * diag
    assert res["outer_iterations"] == ref["outer_iterations"]


# ---- B. off the surface, far out --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [1000.0, 10000.0])
def test_queries_off_a_far_panel(engine, oracle, offset):
    tgt = shifted(synth.panel_points(30_000, 23), offset)
    q = off_surface_queries(offset)
    reset(engine)
    engine.set_target(tgt)
    name = f"B panel {offset:g} m"
    check_nn1(engine, oracle, tgt, q, name, far=True)
    T = rigid(tgt.astype(np.float64).mean(0), 0.01, (0.05, -0.02, 0.03))
    check_nn1(engine, oracle, tgt, q, name + " moved", T=T, far=True)
    engine.set_source(q)
    check_fitness(engine, oracle, q, tgt, EYE, name, far=True)
    check_fitness(engine, oracle, q, tgt, T, name + " moved", far=True)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", [0.0, 0.01])
def test_distant_queries_to_a_panel_at_the_origin(engine, oracle, cell):
    """the grid's margin is relative to the indexed cloud (|x| <= 4 m), the queries are 100 m to 10 km away"""
    tgt = synth.panel_points(30_000, 24)
    q = distant_queries()
    reset(engine, cell_size=cell)
    engine.set_target(tgt)
    name = f"B distant queries cell={cell}"
    check_nn1(engine, oracle, tgt, q, name, far=True)
    engine.set_source(q)
    check_fitness(engine, oracle, q, tgt, EYE, name, far=True)
    T = rigid((0.0, 0.0, 0.0), 0.003, (0.5, -0.2, 0.1))
    check_fitness(engine, oracle, q, tgt, T, name + " moved", far=True)


# ---- C. exact ties ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1024.0])
def test_lattice_midpoints_take_the_lowest_index(engine, oracle, offset):
    tgt = lattice(offset)
    src, ties = midpoints(offset)
    name = f"C midpoints {offset:g}"
    for fp32 in (0, 1):
        reset(engine, mahalanobis_fp32=fp32)
        engine.set_clouds(tgt, src)
        check_correspondences(engine, oracle, src, tgt, EYE, 0.04, False, fp32, name)
        got = check_correspondences(engine, oracle, src, tgt, EYE, 0.04, True, fp32, name)
        assert got[0] == len(src)
        check_fitness(engine, oracle, src, tgt, EYE, name + " seeded")
        check_cost(engine, oracle, src, tgt, got, name)
    check_nn1(engine, oracle, tgt, src, name)
    check_nn1(engine, oracle, tgt, src, name, max_dist=0.04)
    idx, _ = engine.nn1(src)
    D = brute(tgt, src)
    lowest = np.array([np.flatnonzero(r == r.min()).min() for r in D])
    assert np.array_equal(idx, lowest)
    print(f"{name}: {np.bincount(ties)[[2, 4, 8]]} sources with 2 / 4 / 8 ties")


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1024.0])
def test_seeded_pass_moves_to_a_lower_index_tie(engine, oracle, offset):
    """first pass 2^-10 towards b: b is the unique match; the seeded pass at identity starts from b, which now ties
    with a: where a has the lower index the pass must move to it"""
    tgt = lattice(offset)
    src, ia, ib = x_edge_midpoints(tgt, offset)
    T = EYE.copy()
    T[0, 3] = 2.0 ** -10
    name = f"C seeded tie {offset:g}"
    for fp32 in (0, 1):
        reset(engine, mahalanobis_fp32=fp32)
        engine.set_clouds(tgt, src)
        first = check_correspondences(engine, oracle, src, tgt, T, 0.04, False, fp32, name)
        assert np.array_equal(first[1], ib)
        second = check_correspondences(engine, oracle, src, tgt, EYE, 0.04, True, fp32, name)
        assert np.array_equal(second[1], np.minimum(ia, ib))
        print(f"{name}: {int((ia < ib).sum())} seeds moved to the lower index")
        check_fitness(engine, oracle, src, tgt, EYE, name + " seeded")
        # and back: the seed is the lower index, the pass under T must leave it for b
        third = check_correspondences(engine, oracle, src, tgt, T, 0.04, True, fp32, name)
        assert np.array_equal(third[1], ib)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_copies_of_target_points(engine, oracle, offset):
    base = shifted(synth.panel_points(6000, 25), offset)
    tgt = with_copies(base, 300, 5, 26)
    rng = np.random.default_rng(27)
    src = np.concatenate([base[:2000], (base[2000:4000].astype(np.float64) + rng.normal(0, 2e-3, (2000, 3)))])
    src = src.astype(np.float32)
    name = f"C copies {offset:g}"
    reset(engine, max_corr_distance=0.04)
    engine.set_clouds(tgt, src)
    check_correspondences(engine, oracle, src, tgt, EYE, 0.04, False, 0, name)
    got = check_correspondences(engine, oracle, src, tgt, EYE, 0.04, True, 0, name)
    check_fitness(engine, oracle, src, tgt, EYE, name)
    check_cost(engine, oracle, src, tgt, got, name)
    check_nn1(engine, oracle, tgt, src, name)
    check_difference(engine, oracle, src, tgt, 0.0, name)


# ---- D. the float boundary ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_float_boundary(engine, oracle, offset):
    tgt, src, want_i, want_d2, by_limit = boundary_set(offset)
    name = f"D boundary {offset:g}"
    reset(engine)
    engine.set_target(tgt)
    for gate in BOUND_GATES + [1e-30]:
        check_nn1(engine, oracle, tgt, src, f"{name} gate {gate}", max_dist=gate)
    for fp32 in (0, 1):
        for gate in BOUND_GATES + [1e-30]:
            reset(engine, max_corr_distance=gate, mahalanobis_fp32=fp32)
            engine.set_clouds(tgt, src)
            first = check_correspondences(engine, oracle, src, tgt, EYE, gate, False, fp32, f"{name} gate {gate}")
            want = want_d2.astype(np.float64) < gate * gate
            assert first[0] == int(want.sum()) and np.array_equal(first[1] >= 0, want)
            got = check_correspondences(engine, oracle, src, tgt, EYE, gate, True, fp32, f"{name} gate {gate}")
            check_cost(engine, oracle, src, tgt, got, f"{name} gate {gate}")
    for thr in BOUND_THRESHOLDS + [0.0, -1.0]:
        check_difference(engine, oracle, src, tgt, thr, name)
    mask, _ = engine.cloud_difference(src, tgt, 0.0)
    assert not mask[want_d2 == 0].any() and mask[want_d2 > 0].all()
    # max_range: the d2 at or just above 0.04^2 exactly, and one attainable value above
    at, above = by_limit[0.04 * 0.04][2:]
    reset(engine)
    engine.set_clouds(tgt, src)
    for mr in (float(at), float(above), 0.0):
        check_fitness(engine, oracle, src, tgt, EYE, f"{name} unseeded", max_range=mr)
    engine.correspondences(EYE)
    for mr in (float(at), float(above), 0.0):
        check_fitness(engine, oracle, src, tgt, EYE, f"{name} seeded", max_range=mr)


# ---- E. non-finite inputs and limits ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nonfinite_pair(panel_pair):
    src, tgt = panel_pair
    return with_nonfinite(src[:20000], seed=6), with_nonfinite(tgt[:20000], seed=7, every=13)


@pytest.mark.gpu
@pytest.mark.parametrize("gate", [0.04, 1.0, np.inf, 0.0, -0.04, np.nan])
def test_nonfinite_rows_and_gates(engine, oracle, nonfinite_pair, gate):
    src, tgt = nonfinite_pair
    T1 = rigid((2.0, 0.0, 0.0), 0.002, (0.003, -0.002, 0.001))
    name = f"E gate {gate}"
    for fp32 in (0, 1):
        reset(engine, max_corr_distance=gate, mahalanobis_fp32=fp32)
        engine.set_clouds(tgt, src)
        check_correspondences(engine, oracle, src, tgt, T1, gate, False, fp32, name)
        got = check_correspondences(engine, oracle, src, tgt, T1, gate, True, fp32, name)
        check_cost(engine, oracle, src, tgt, got, name)
    check_nn1(engine, oracle, tgt, src, name, T=T1, max_dist=gate if np.isfinite(gate) else 0.0)


@pytest.mark.gpu
def test_nan_gate_align_finds_too_few_pairs(engine, oracle, cube_pair):
    """PCL compares d2 < NaN: no pair, NotEnoughPointsException, hasConverged() false"""
    from oracle.oracle import default_params
    src, tgt, _ = cube_pair
    ref = oracle.align(src, tgt, default_params(max_corr_distance=float("nan")))
    assert ref["converged"] == 0 and ref["n_pairs_last"] == 0
    reset(engine, max_corr_distance=float("nan"))
    engine.set_clouds(tgt, src)
    res = engine.align(raise_on_failure=False)
    assert res["rc"] == E_NOT_ENOUGH_CORRESPONDENCES and res["converged"] == 0 and res["corr_pairs_last"] == 0
    assert np.array_equal(res["transform"], EYE)
    ms, _ = engine.bench_kernel(2, EYE, iters=1)          # the NN pass of the kernel benchmark takes the same gate
    assert ms >= 0.0
    reset(engine)


@pytest.mark.gpu
@pytest.mark.parametrize("max_range", [None, 1e-4, np.nan, 0.0, -1.0, np.inf])
def test_nonfinite_rows_fitness(engine, oracle, nonfinite_pair, max_range):
    src, tgt = nonfinite_pair
    T1 = rigid((2.0, 0.0, 0.0), 0.002, (0.003, -0.002, 0.001))
    reset(engine, max_corr_distance=1.0)
    engine.set_clouds(tgt, src)
    check_fitness(engine, oracle, src, tgt, T1, "E unseeded", max_range=max_range)
    engine.correspondences(T1)
    check_fitness(engine, oracle, src, tgt, T1, "E seeded", max_range=max_range)


DIFF_LIMITS = [4e-4, np.nan, np.inf, 1e300, FLT_MAX, 0.0, -1.0, -np.inf]


@pytest.mark.gpu
@pytest.mark.parametrize("thr", DIFF_LIMITS)
def test_nonfinite_rows_difference(engine, oracle, nonfinite_pair, thr):
    src, tgt = nonfinite_pair
    reset(engine)
    check_difference(engine, oracle, src, tgt, thr, "E")
    check_difference(engine, oracle, src[:3000], src, thr, "E self")
    # the split calls: one subtract index, several runs
    engine.difference_set_subtract(tgt)
    mask, kept = engine.difference_run(src, thr)
    om, ok = oracle.difference(src, tgt[finite_rows(tgt)], thr)
    assert np.array_equal(mask, om) and kept == ok


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [np.nan, np.inf, 4e-4, -1.0])
def test_group_difference_limits(oracle, nonfinite_pair, thr):
    """gicpb_group_cloud_difference takes the same limits: its subtract window's halo is the search radius"""
    from leica_point_cloud_processing_b200 import EngineGroup
    src, tgt = nonfinite_pair
    grp = EngineGroup([0, 0])
    try:
        mask, kept = grp.cloud_difference(src, tgt, thr)
    finally:
        grp.close()
    om, ok = oracle.difference(src, tgt[finite_rows(tgt)], thr)
    print(f"E group difference thr={thr!r}: kept {kept} (oracle {ok})")
    assert np.array_equal(mask, om) and kept == ok


@pytest.mark.gpu
def test_clouds_without_a_finite_point_are_refused(engine, cube_pair):
    from leica_point_cloud_processing_b200 import GicpError
    src, tgt, _ = cube_pair
    empty = np.full((50, 3), np.nan, np.float32)
    empty[::3, 1] = np.inf
    reset(engine)
    with pytest.raises(GicpError) as e:
        engine.set_target(empty)
    assert e.value.code == E_BADARG
    with pytest.raises(GicpError) as e:
        engine.cloud_difference(src, empty, 4e-4)
    assert e.value.code == E_BADARG
    # the context is still usable
    mask, kept = engine.cloud_difference(src, tgt, 4e-4)
    assert kept == int(mask.sum())


# ---- F. scale ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_million_points_1_km_out(engine, fast_oracle):
    src, tgt = outlier_pair(1 << 20, 1000.0, 40)
    c = tgt.astype(np.float64).mean(0)
    T1 = rigid(c, 0.001, (0.002, -0.001, 0.001))
    T2 = rigid(c, 0.0012, (0.0022, -0.0008, 0.001))
    gate = 1.0
    with timed("F 1 M pair 1 km out"):
        for fp32 in (0, 1):
            reset(engine, max_corr_distance=gate, mahalanobis_fp32=fp32)
            engine.set_clouds(tgt, src)
            check_correspondences(engine, fast_oracle, src, tgt, T1, gate, False, fp32, "F 1 M", far=True)
            check_correspondences(engine, fast_oracle, src, tgt, T2, gate, True, fp32, "F 1 M")
        check_fitness(engine, fast_oracle, src, tgt, T2, "F 1 M seeded")
        for thr in (4e-4, 1.2e-2):
            check_difference(engine, fast_oracle, src, tgt, thr, "F 1 M")
