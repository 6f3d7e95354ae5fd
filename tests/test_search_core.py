"""CPU checks of the product's search logic (mulls_b200/csrc/search_core.cuh, __host__ __device__): the very functions
k_search runs on the device (walk_greedy_seed, nn_search_walk) are instantiated on the host by
tests/harness/search_host.cu (grid built there with the same keys / hash / entry layout as k_hash_build) and compared
with a brute-force scan under the reference's total order (FLANN float distance, then original index) and with the
oracle's kd-tree NN (cregistration.hpp:1742-1745)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from mulls_b200 import synth
from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    src = os.path.join(ROOT, "tests", "harness", "search_host.cu")
    out = os.path.join(ROOT, "tests", "harness", "_build", "libsearch_host.so")
    deps = [src] + [os.path.join(ROOT, "mulls_b200", "csrc", f) for f in ("search_core.cuh", "grid_key.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20014,20011",
                               "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-o", out, src])
    lb = C.CDLL(out)
    lb.sh_build.restype = C.c_void_p
    lb.sh_build.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int]
    lb.sh_free.argtypes = [C.c_void_p]
    lb.sh_search.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_int, C.c_float, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_void_p]
    lb.sh_search_cert.argtypes = lb.sh_search.argtypes + [C.c_void_p]
    lb.sh_levels_for.restype = C.c_int
    lb.sh_levels_for.argtypes = [C.c_float, C.c_float, C.c_float, C.c_float, C.c_int]
    lb.sh_h0_for.restype = C.c_float
    lb.sh_h0_for.argtypes = [C.c_double, C.c_float]
    lb.sh_morton_roundtrip.restype = C.c_uint32
    lb.sh_morton_roundtrip.argtypes = [C.c_uint32]
    return lb


def run(lib, tgt_xyz, q_xyz, radius, seeds=None, leaf=32, h0=0.125, reseed=-1.0, mode=0, want_cert=False, levels=None):
    """search every query within `radius` on a grid of level-0 cell size h0; `levels` defaults to what k_pair_setup
    chooses when `radius` is the largest radius of the pair (2.5 x dis_thre_unit, a shrinking schedule)"""
    tgt_xyz = np.ascontiguousarray(tgt_xyz, np.float32)
    q_xyz = np.ascontiguousarray(q_xyz, np.float32)
    origin = (tgt_xyz.min(0) - 2 * h0).astype(np.float32)
    pts4 = np.ascontiguousarray(np.concatenate([tgt_xyz, np.zeros((len(tgt_xyz), 1), np.float32)], axis=1))
    G = lib.sh_build(pts4.ctypes.data, len(tgt_xyz), float(origin[0]), float(origin[1]), float(origin[2]), h0,
                     levels if levels is not None else lib.sh_levels_for(h0, radius / 2.5, 0.0, 2.0, 1), leaf)
    m = len(q_xyz)
    idx = np.empty(m, np.int32)
    d2 = np.empty(m, np.float32)
    stats = np.zeros(12, np.uint64)
    stats[10] = mode  # 1: the small cells of a block are queued and examined together (k_search's late iterations)
    r = np.float32(radius)
    r2 = np.float32(np.float32(np.float64(r) * np.float64(r)) * np.float32(1.0001))
    sd = np.ascontiguousarray(seeds, np.int32) if seeds is not None else None
    cert = np.empty(m, np.float32)
    lib.sh_search_cert(G, q_xyz.ctypes.data, sd.ctypes.data if sd is not None else None, m, float(r2), 5, float(reseed),
                       idx.ctypes.data, d2.ctypes.data, stats.ctypes.data, None, cert.ctypes.data)
    lib.sh_free(G)
    return (idx, d2, cert) if want_cert else (idx, d2)


def brute(tgt_xyz, q_xyz):
    """argmin under (float32 FLANN distance, index)."""
    t = np.asarray(tgt_xyz, np.float32)
    out_i = np.empty(len(q_xyz), np.int32)
    out_d = np.empty(len(q_xyz), np.float32)
    for k, p in enumerate(np.asarray(q_xyz, np.float32)):
        d = t - p
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]  # float32 throughout, FLANN's order
        j = int(np.argmin(d2))  # first minimum = lowest index
        out_i[k], out_d[k] = j, d2[j]
    return out_i, out_d


def check(idx, d2, bi, bd, radius):
    r2 = np.float64(np.float32(radius)) ** 2
    inside = bd.astype(np.float64) <= r2
    assert np.array_equal(idx[inside], bi[inside])
    assert np.array_equal(d2[inside], bd[inside])
    # a query with nothing inside the radius may report a farther seed or nothing: k_search's keep test drops it
    out = ~inside
    assert np.all((idx[out] < 0) | (d2[out].astype(np.float64) > r2))


def test_morton_roundtrip(lib):
    for v in list(range(0, 4096, 7)) + [4095]:
        assert lib.sh_morton_roundtrip(v) == 1


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_clouds_equal_brute_force(lib, seed):
    rng = np.random.default_rng(seed)
    # clustered planar + uniform clutter, with exact duplicates and equidistant pairs (ties -> lowest index)
    plane = np.c_[rng.uniform(-20, 20, 4000), rng.uniform(-20, 20, 4000), rng.normal(0, 0.02, 4000)]
    wall = np.c_[rng.uniform(-20, 20, 3000), np.full(3000, 7.5) + rng.normal(0, 0.02, 3000), rng.uniform(0, 6, 3000)]
    dense = rng.normal(0, 0.15, (3000, 3)) + [3.0, 2.0, 0.5]
    tgt = np.concatenate([plane, wall, dense, plane[:200], dense[:100]]).astype(np.float32)  # duplicates
    q = np.concatenate([tgt[rng.integers(0, len(tgt), 1500)] + rng.normal(0, 0.05, (1500, 3)),
                        rng.uniform(-25, 25, (500, 3)), tgt[:300]]).astype(np.float32)
    bi, bd = brute(tgt, q)
    for radius in (3.5, 1.25, 0.3):
        for leaf in (32, 4):
            for mode in (0, 1):
                idx, d2 = run(lib, tgt, q, radius, leaf=leaf, mode=mode)
                check(idx, d2, bi, bd, radius)
    # seeded: good seeds (the answer), stale seeds (random target), mixed with none
    seeds = bi.copy()
    seeds[::3] = rng.integers(0, len(tgt), len(seeds[::3]))
    seeds[1::7] = -1
    for reseed in (-1.0, 0.0625):
        for mode in (0, 1):
            idx, d2 = run(lib, tgt, q, 3.5, seeds=seeds, reseed=reseed, mode=mode)
            check(idx, d2, bi, bd, 3.5)


def test_tiny_and_degenerate_grids(lib):
    tgt = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    q = np.array([[0.4, 0.1, 0], [0.5, 0, 0], [10, 10, 10], [0, 0, 0]], np.float32)
    bi, bd = brute(tgt, q)
    idx, d2 = run(lib, tgt, q, 3.5)
    check(idx, d2, bi, bd, 3.5)
    assert idx[1] == 0  # equidistant to targets 0 and 1: the lower index
    # all targets in one spot (one cell at every level, count > leaf_count)
    tgt = np.tile(np.array([[2.0, 2.0, 2.0]], np.float32), (100, 1))
    idx, d2 = run(lib, tgt, q, 3.5, leaf=8)
    bi, bd = brute(tgt, q)
    check(idx, d2, bi, bd, 3.5)


def test_synthetic_pair_equals_oracle_kdtree(lib):
    """every class of the 'small' synthetic pair, unseeded and seeded with a moved cloud's previous answer"""
    pair = synth.make_pair(1000, "small")
    for c in range(6):
        tgt, src = pair["tgt"][c], pair["src"][c]
        if len(tgt) < 3 or len(src) < 3:
            continue
        oi, od = oracle.nn(tgt, src, 1e9)
        for mode in (0, 1):
            idx, d2 = run(lib, tgt[:, :3], src[:, :3], 3.5, mode=mode)
            check(idx, d2, oi, od, 3.5)
        moved = src.copy()
        moved[:, 0] += 0.07
        moved[:, 1] -= 0.03
        oi2, od2 = oracle.nn(tgt, moved, 1e9)
        idx2, d22 = run(lib, tgt[:, :3], moved[:, :3], 1.25, seeds=oi, reseed=0.0625)
        check(idx2, d22, oi2, od2, 1.25)


def second_nearest_sq(tgt_xyz, q_xyz, best):
    """exact (float64) squared distance of the closest target other than `best` (or of the closest, where best < 0)"""
    t = np.asarray(tgt_xyz, np.float64)
    out = np.empty(len(q_xyz))
    for k, p in enumerate(np.asarray(q_xyz, np.float64)):
        d2 = ((t - p) ** 2).sum(1)
        if best[k] >= 0:
            d2[best[k]] = np.inf
        out[k] = d2.min()
    return out


@pytest.mark.parametrize("seed", [4, 5])
def test_certificate_is_a_lower_bound_on_every_other_target(lib, seed):
    """nn_search_walk's return value: no target other than the answer is closer than it — what lets k_search keep a
    match in a later iteration without searching (|p - q| + movement < certificate)."""
    rng = np.random.default_rng(seed)
    plane = np.c_[rng.uniform(-20, 20, 5000), rng.uniform(-20, 20, 5000), rng.normal(0, 0.02, 5000)]
    wall = np.c_[rng.uniform(-20, 20, 3000), np.full(3000, 7.5) + rng.normal(0, 0.02, 3000), rng.uniform(0, 6, 3000)]
    dense = rng.normal(0, 0.15, (3000, 3)) + [3.0, 2.0, 0.5]
    tgt = np.concatenate([plane, wall, dense, plane[:100]]).astype(np.float32)
    q = np.concatenate([tgt[rng.integers(0, len(tgt), 2000)] + rng.normal(0, 0.05, (2000, 3)),
                        rng.uniform(-25, 25, (500, 3))]).astype(np.float32)
    bi, _ = brute(tgt, q)
    for radius in (3.5, 0.6):
        for leaf in (32, 4):
            for mode in (0, 1):
                for seeds in (None, bi):
                    idx, d2, cert = run(lib, tgt, q, radius, seeds=seeds, leaf=leaf, mode=mode, want_cert=True)
                    others = second_nearest_sq(tgt, q, idx)
                    assert np.all(cert.astype(np.float64) <= others * (1 + 1e-5) + 1e-9)
                    useful = (idx >= 0) & (cert > d2 * 1.05)
                    assert useful.mean() > 0.3  # and it is not vacuous: a real margin for a good share of the queries


def test_a_kept_match_equals_a_fresh_search(lib):
    """the skip rule of k_search on the host: queries move a little; where |p' - q| + |p' - p| stays below the
    certificate the previous match must be what a fresh search (and brute force) returns"""
    rng = np.random.default_rng(11)
    pair = synth.make_pair(1000, "small")
    tgt, src = pair["tgt"][0][:, :3], pair["src"][0][:, :3]
    idx, d2, cert = run(lib, tgt, src, 1.5, want_cert=True)
    kept_total = 0
    for step in (0.002, 0.01, 0.05):
        moved = (src + rng.normal(0, step, src.shape)).astype(np.float32)
        bi, bd = brute(tgt, moved)
        m = idx >= 0
        d1 = np.sqrt(((moved[m].astype(np.float64) - tgt[idx[m]].astype(np.float64)) ** 2).sum(1))
        delta = np.sqrt(((moved[m].astype(np.float64) - src[m].astype(np.float64)) ** 2).sum(1))
        keep = (d1 + delta) * 1.0001 + 3e-5 < np.sqrt(cert[m].astype(np.float64)) * 0.9999
        assert np.array_equal(bi[m][keep], idx[m][keep])
        kept_total += int(keep.sum())
    assert kept_total > 0.5 * len(src)


def test_points_on_cell_boundaries_and_queries_outside_the_grid(lib):
    """coordinates that are exact multiples of the cell size (every point sits on a cell boundary of every level), queries
    on boundaries, far outside the grid, and at huge coordinates: answers = brute force, certificates stay lower bounds"""
    h0 = 0.125
    ax = np.arange(0, 24, dtype=np.float32) * np.float32(h0 / 2)  # lattice at half the cell size
    gx, gy, gz = np.meshgrid(ax, ax, ax[:6], indexing="ij")
    tgt = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], axis=1).astype(np.float32)
    rng = np.random.default_rng(21)
    q = np.concatenate([
        tgt[rng.integers(0, len(tgt), 300)],                                             # on targets (distance 0, many ties around)
        tgt[rng.integers(0, len(tgt), 300)] + np.float32(h0 / 4),                        # cell centres of the fine lattice: 8-way ties
        (rng.integers(-8, 40, (300, 3)) * np.float32(h0)).astype(np.float32),            # on level-0 boundaries, partly outside
        rng.uniform(-30, 30, (200, 3)).astype(np.float32),                               # far outside the grid
        np.array([[1e4, 1e4, 1e4], [-1e4, 0, 0], [0.7, 0.7, 400.0]], np.float32)]).astype(np.float32)
    bi, bd = brute(tgt, q)
    for radius in (3.5, 0.2, 0.05):
        for leaf in (32, 2):
            for mode in (0, 1):
                idx, d2, cert = run(lib, tgt, q, radius, leaf=leaf, mode=mode, want_cert=True)
                check(idx, d2, bi, bd, radius)
                others = second_nearest_sq(tgt, q, idx)
                assert np.all(cert.astype(np.float64) <= others * (1 + 1e-5) + 1e-9)
    # seeded with the answers and with wrong seeds
    seeds = bi.copy()
    seeds[::2] = rng.integers(0, len(tgt), len(seeds[::2]))
    idx, d2 = run(lib, tgt, q, 3.5, seeds=seeds, reseed=0.0625)
    check(idx, d2, bi, bd, 3.5)


def test_single_dense_spot_with_a_stack_too_small_to_split_it(lib):
    """thousands of points inside one level-0 cell next to a sparse halo: level-0 cells are scanned whatever they hold, and a
    dense cell that cannot be split any further (stack full) is scanned as a whole — still exact"""
    rng = np.random.default_rng(5)
    dense = (rng.uniform(0, 0.1, (5000, 3)) + [1.0, 1.0, 1.0]).astype(np.float32)
    halo = rng.uniform(-3, 5, (2000, 3)).astype(np.float32)
    tgt = np.concatenate([dense, halo])
    q = np.concatenate([dense[::50] + np.float32(0.001), halo[::10] + np.float32(0.01), rng.uniform(0.9, 1.2, (200, 3)).astype(np.float32)])
    bi, bd = brute(tgt, q)
    for leaf in (32, 1):
        idx, d2, cert = run(lib, tgt, q, 3.5, leaf=leaf, want_cert=True)
        check(idx, d2, bi, bd, 3.5)
        assert np.all(cert.astype(np.float64) <= second_nearest_sq(tgt, q, idx) * (1 + 1e-5) + 1e-9)
