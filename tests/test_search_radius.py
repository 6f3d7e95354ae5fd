"""CPU checks of the search at every radius a pair searches with and on every grid shape k_pair_setup builds: the
product's nn_search_walk (search_core.cuh, instantiated on the host by tests/harness/search_host.cu) on grids sized by
the product's own rules (grid_h0, grid_levels: sh_h0_for, sh_levels_for), against a brute-force scan under the
reference's total order (FLANN float distance, then original index) and a float64 scan; the certificate each search
returns must stay a lower bound on the distance of every other target."""
import numpy as np
import pytest

from test_search_core import lib, run  # noqa: F401  (lib: the harness fixture)

H0_MIN = 0.125  # the default h0_min of a context


def schedule(unit, tmin, rate, max_iter):
    """thresholds of iterations 0 .. max_iter-1 as solve_and_advance computes them (float state, double update)"""
    out, thre = [], np.float32(unit)
    for _ in range(max_iter):
        out.append(thre)
        t = np.float64(thre) / np.float64(np.float32(rate))
        thre = np.float32(t) if t > np.float64(np.float32(tmin)) else np.float32(tmin)
    return out


def search_radius(thre):
    """k_search's radius: 2.5 * thre in float (its square is kept in double, its pruning bound is 1.0001 x that)"""
    return float(np.float32(2.5) * np.float32(thre))


def reference(tgt, q, chunk=256):
    """per query: brute force under the reference's total order (float32 FLANN distance, FLANN's summation order, ties
    to the lower index), and the float64 squared distances of the two nearest targets with the index of the nearest"""
    t32, q32 = np.asarray(tgt, np.float32), np.asarray(q, np.float32)
    t64, q64 = t32.astype(np.float64), q32.astype(np.float64)
    n = len(q32)
    bi, bd = np.empty(n, np.int64), np.empty(n, np.float32)
    j64, m1, m2 = np.empty(n, np.int64), np.empty(n), np.empty(n)
    for s in range(0, n, chunk):
        d = t32[None, :, :] - q32[s:s + chunk, None, :]
        f = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        bi[s:s + chunk] = np.argmin(f, axis=1)  # first minimum = lowest index
        bd[s:s + chunk] = f[np.arange(len(f)), bi[s:s + chunk]]
        e = ((t64[None, :, :] - q64[s:s + chunk, None, :]) ** 2).sum(-1)
        j = np.argmin(e, axis=1)
        j64[s:s + chunk] = j
        m1[s:s + chunk] = e[np.arange(len(e)), j]
        e[np.arange(len(e)), j] = np.inf
        m2[s:s + chunk] = e.min(axis=1) if e.shape[1] > 1 else np.inf
    return bi, bd, j64, m1, m2


def check_exact(ref, radius, idx, d2, cert, tgt, q):
    """answers = brute force inside the radius, no float64-closer target beyond rounding, certificate a lower bound"""
    bi, bd, j64, m1, m2 = ref
    r2 = np.float64(np.float32(radius)) ** 2
    inside = bd.astype(np.float64) <= r2
    bad = np.flatnonzero(inside & ((idx != bi) | (d2 != bd)))
    assert len(bad) == 0, f"{len(bad)} of {inside.sum()} answers differ from brute force, e.g. query {q[bad[0]]}: " \
                          f"{idx[bad[0]]} / {d2[bad[0]]} instead of {bi[bad[0]]} / {bd[bad[0]]}"
    out = ~inside
    assert np.all((idx[out] < 0) | (d2[out].astype(np.float64) > r2))
    # float64: the answer is the nearest target up to rounding (an answer beyond the radius is dropped by k_search)
    t64, q64 = np.asarray(tgt, np.float64), np.asarray(q, np.float64)
    e_ans = ((t64[idx[inside]] - q64[inside]) ** 2).sum(1)
    assert np.all(e_ans <= m1[inside] * (1 + 1e-6) + 1e-10)
    # the certificate bounds every target other than the answer from below (second_nearest_sq of test_search_core)
    others = np.where(idx == j64, m2, m1)
    dup = (idx >= 0) & (idx != j64)  # the answer is an exact tie of the float64 nearest: the nearest is another target
    others[dup] = np.minimum(m1[dup], ((t64[idx[dup]] - q64[dup]) ** 2).sum(1))
    assert np.all(cert.astype(np.float64) <= others * (1 + 1e-5) + 1e-9)
    return int(inside.sum())


# (dis_thre_unit, dis_thre_min, dis_thre_update_rate, max_iter_num): the shrinking default, and every parameter set of
# the reference's call sites (SURVEY Appendix C), with the level count each gives at h0 = 0.125 and 0.25
APPENDIX_C = [
    ((1.5, 0.4, 1.1, 20), 7, 6),    # mulls_icp_default_params
    ((3.0, 0.75, 1.1, 10), 8, 7),   # test/mulls_reg.cpp:194-195 (run script values)
    ((1.4, 0.5, 1.1, 20), 7, 6),    # test/mulls_slam.cpp:642-648 / 679-685, first scan (add_length 0)
    ((2.4, 0.5, 1.1, 20), 8, 7),    # the same with add_length 1.0
    ((2.25, 0.6, 1.1, 3), 8, 7),    # test/mulls_slam.cpp:477-482: 1.5 x the defaults, 3 iterations
    ((5.25, 0.8, 1.1, 3), 9, 8),    # test/mulls_slam.cpp:560-566: 3.5 x / 2.0 x
    ((2.1, 0.75, 1.1, 3), 8, 7),    # the map-to-map variant of test_gpu_parity
]


def test_level_rule_keeps_the_shrinking_schedules_and_grows_with_the_threshold(lib):
    for (unit, tmin, rate, iters), l125, l25 in APPENDIX_C:
        assert lib.sh_levels_for(0.125, unit, tmin, rate, iters) == l125
        assert lib.sh_levels_for(0.25, unit, tmin, rate, iters) == l25
        # = the level count of iteration 0's radius alone: the schedule only shrinks
        assert lib.sh_levels_for(0.125, unit, tmin, rate, iters) == lib.sh_levels_for(0.125, unit, 0.0, 2.0, 1)
    # src/build_pose_graph.cpp:447-453: dis_thre_min = 2 * nonground_downsample_rate * vf_downsample_resolution_als
    # is not compared with reg_corr_dis_thre — a threshold that rises to dis_thre_min after the first iteration
    assert lib.sh_levels_for(0.125, 1.5, 4.0, 1.1, 20) == 9 > lib.sh_levels_for(0.125, 1.5, 0.4, 1.1, 20)
    assert lib.sh_levels_for(0.125, 1.5, 4.0, 1.1, 1) == 7  # one iteration searches with dis_thre_unit only
    assert lib.sh_levels_for(0.125, 1.5, 0.4, 0.8, 10) == 10  # 1.5 / 0.8^9 = 11.2 m
    assert lib.sh_levels_for(0.125, 1.5, 0.4, 0.8, 40) == 12  # beyond the full pyramid: capped
    assert lib.sh_levels_for(0.125, 1.5, 0.4, 1.0, 20) == 7
    assert lib.sh_levels_for(0.125, 1.5, 3.0, 1.0, 20) == 8
    # the doubling rule of the level-0 cell size
    for ext, h0 in ((100.0, 0.125), (505.0, 0.125), (515.0, 0.25), (600.0, 0.25), (1500.0, 0.5), (3000.0, 1.0)):
        assert lib.sh_h0_for(ext, H0_MIN) == h0


def run_schedule(lib, tgt, q, h0, sched, leaf=32):
    unit, tmin, rate, iters = sched
    L = lib.sh_levels_for(h0, unit, tmin, rate, iters)
    n_inside = 0
    ref = reference(tgt, q)
    for thre in sorted(set(schedule(unit, tmin, rate, iters))):
        radius = search_radius(thre)
        for mode in (0, 1):
            idx, d2, cert = run(lib, tgt, q, radius, leaf=leaf, h0=h0, mode=mode, want_cert=True, levels=L)
            n_inside += check_exact(ref, radius, idx, d2, cert, tgt, q)
    return L, n_inside


@pytest.mark.parametrize("sched", [(1.5, 0.4, 0.8, 10), (1.5, 0.4, 0.95, 20), (1.5, 3.0, 1.0, 6), (1.5, 4.0, 1.1, 5)],
                         ids=["rate0.8", "rate0.95", "rate1_min3", "min4"])
def test_radius_above_the_first_iterations_sizing(lib, sched):
    """thresholds that grow (rate <= 1, or dis_thre_min > dis_thre_unit): sparse targets, so that most nearest targets lie
    beyond the coverage of a grid sized for 2.5 x dis_thre_unit"""
    rng = np.random.default_rng(31)
    tgt = rng.uniform(0, 80, (800, 3)).astype(np.float32)
    q = rng.uniform(-5, 85, (1500, 3)).astype(np.float32)
    L, n_inside = run_schedule(lib, tgt, q, 0.125, sched)
    assert L > lib.sh_levels_for(0.125, 1.5, 0.0, 2.0, 1)
    assert n_inside > 1000


def test_radius_beyond_the_full_pyramid(lib):
    """thre up to 60 m at h0 0.125: 2.5 x thre exceeds the coverage of the top level's 2x2x2 block (128 m), so the top
    level must walk the whole grid — queries in all four quarters of the top level along every axis, and outside the grid"""
    rng = np.random.default_rng(32)
    # the grid spans ~512 m (an anchor at two corners): its top level is 2 x 2 x 2 cells of 256 m. Decoys: along each
    # axis, queries in an outer quarter of the top level (within 128 m of the grid's face) whose only targets within
    # 170 m are a small cluster across the middle plane, 140-160 m away — outside the 2x2x2 block of their own level-10
    # cell's side, which reaches the middle plane only from the inner quarters
    queries, clusters = [], []

    def dmin(a, b):
        return np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)).min() if len(b) else np.inf

    for axis in range(3):
        for lo_side in (True, False):
            placed = 0
            while placed < 1:  # one decoy group per axis and side, clear of the other groups
                c = np.empty(3)
                c[[k for k in range(3) if k != axis]] = rng.uniform(20, 485, 2)
                qx, tx = (120.0, 265.0) if lo_side else (385.0, 240.0)
                qa, ta = c.copy(), c.copy()
                qa[axis], ta[axis] = qx, tx
                cl, qs = ta + rng.uniform(-3, 3, (20, 3)), qa + rng.uniform(-2, 2, (10, 3))
                if dmin(cl, np.concatenate(queries or [np.empty((0, 3))])) > 170 and \
                        dmin(qs, np.concatenate(clusters or [np.empty((0, 3))])) > 170:
                    queries.append(qs)
                    clusters.append(cl)
                    placed += 1
    corners = np.array([[0, 0, 0], [505, 505, 505]])
    decoy_q = np.concatenate(queries)
    spread = rng.uniform(0, 505, (300, 3))
    far = np.sqrt(((spread[:, None, :] - decoy_q[None]) ** 2).sum(-1)).min(1) > 170.0
    tgt = np.concatenate([corners, spread[far]] + clusters).astype(np.float32)
    # queries: the decoys, uniform over the grid and beyond, and next to the top-level split planes
    q = np.concatenate([decoy_q, rng.uniform(-40, 545, (1500, 3)),
                        np.c_[rng.choice([120.0, 130.0, 250.0, 262.0, 380.0, 390.0], 500), rng.uniform(0, 505, (500, 2))]
                        ]).astype(np.float32)
    bd = reference(tgt, decoy_q)[1].astype(np.float64)
    assert np.all((bd > 128.0 ** 2) & (bd < 165.0 ** 2))  # beyond the 2x2x2 block, inside the radius
    sched = (1.5, 0.4, 0.8, 18)  # 1.5 / 0.8^17 = 66.6 m
    assert max(schedule(*sched)) > 60.0
    L, n_inside = run_schedule(lib, tgt, q, 0.125, sched)
    assert L == 12
    assert n_inside > 2000


@pytest.mark.parametrize("extent", [600.0, 1500.0, 3000.0])
def test_wide_clouds(lib, extent):
    """clouds wide enough to double h0 (k_pair_setup's rule), radii 0.3 / 3.5 / 10 m, small and large leaves"""
    rng = np.random.default_rng(int(extent))
    n = 12000
    ground = np.c_[rng.uniform(0, extent, n), rng.uniform(0, extent, n), rng.normal(0, 0.05, n)]
    poles = np.repeat(rng.uniform(0, extent, (200, 2)), 20, axis=0)
    poles = np.c_[poles + rng.normal(0, 0.03, poles.shape), rng.uniform(0, 8, len(poles))]
    tgt = np.concatenate([ground, poles, [[extent, extent, 30.0]]]).astype(np.float32)
    q = np.concatenate([tgt[rng.integers(0, len(tgt), 1200)] + rng.normal(0, 0.3, (1200, 3)),
                        rng.uniform(-20, extent + 20, (600, 3)) * [1, 1, 0.02],
                        rng.uniform(-100, extent + 100, (100, 3))]).astype(np.float32)
    ext = float(np.max(tgt.max(0).astype(np.float64) - tgt.min(0).astype(np.float64)))
    h0 = lib.sh_h0_for(ext, H0_MIN)
    assert h0 == {600.0: 0.25, 1500.0: 0.5, 3000.0: 1.0}[extent]
    ref = reference(tgt, q)
    for radius in (0.3, 3.5, 10.0):
        L = lib.sh_levels_for(h0, radius / 2.5, 0.0, 2.0, 1)
        for leaf in (32, 2):
            idx, d2, cert = run(lib, tgt, q, radius, leaf=leaf, h0=h0, want_cert=True, levels=L)
            check_exact(ref, radius, idx, d2, cert, tgt, q)


@pytest.mark.parametrize("offset", [(5000.0, -3000.0, 0.0), (50000.0, 50000.0, -50000.0), (4090.0, 8185.0, 2040.0)],
                         ids=["5km", "50km", "binade_edges"])
def test_far_from_the_origin(lib, offset):
    """the boundary lattice of test_points_on_cell_boundaries_and_queries_outside_the_grid, far from the origin (the
    last offset puts the grid across 4096 / 8192 / 2048 m, where the cell walls' float coordinates change ulp):
    queries on targets and on cell boundaries, each nudged by +-1 ulp"""
    h0 = 0.125
    ax = np.arange(0, 24, dtype=np.float32) * np.float32(h0 / 2)
    gx, gy, gz = np.meshgrid(ax, ax, ax[:6], indexing="ij")
    base = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], axis=1)
    off = np.asarray(offset, np.float32)
    tgt = (base + off).astype(np.float32)
    rng = np.random.default_rng(22)
    on_t = tgt[rng.integers(0, len(tgt), 300)]
    on_b = ((rng.integers(-8, 40, (300, 3)) * np.float32(h0)).astype(np.float32) + off).astype(np.float32)
    on_c = (tgt[rng.integers(0, len(tgt), 200)] + np.float32(h0 / 4)).astype(np.float32)
    q = [on_t, on_b, on_c]
    for pts in (on_t, on_b):
        for direction in (np.inf, -np.inf):
            nudged = pts.copy()
            axis = rng.integers(0, 3, len(pts))
            nudged[np.arange(len(pts)), axis] = np.nextafter(pts[np.arange(len(pts)), axis], np.float32(direction))
            q.append(nudged)
            q.append(np.nextafter(pts, np.float32(direction)))  # every coordinate
    q.append((rng.uniform(-5, 7, (200, 3)) + off).astype(np.float32))
    q = np.concatenate(q).astype(np.float32)
    ref = reference(tgt, q)
    for radius in (3.5, 0.2, 0.05):
        for leaf in (32, 2):
            for mode in (0, 1):
                idx, d2, cert = run(lib, tgt, q, radius, leaf=leaf, h0=h0, mode=mode, want_cert=True)
                check_exact(ref, radius, idx, d2, cert, tgt, q)
