"""GPU checks of the correspondence search at the edges of its grid: threshold schedules whose radius grows past the
first iteration's (dis_thre_update_rate <= 1, dis_thre_min > dis_thre_unit) against the oracle through all three
iteration drivers; the device-built grid (k_hash_build, k_hash_layout, per-pair h0 / n_levels) against brute force
through mulls_nn_query on wide, offset, lattice and dense clouds under non-default grid tunables; and a batch of pairs
whose grids differ, each bit-identical to the same pair run alone."""
import numpy as np
import pytest

from mulls_b200 import abi, synth
from test_gpu_parity import assert_parity

DEFAULTS = {"loop_kernel": 1, "use_graph": 1, "leaf_count": 32, "hash_slack": 4, "h0_min_mm": 125}
DRIVERS = [{"loop_kernel": 1, "use_graph": 1},   # the cooperative k_icp_loop
           {"loop_kernel": 0, "use_graph": 1},   # the CUDA graph
           {"loop_kernel": 0, "use_graph": 0}]   # the host launch loop
N_DECOYS = 30


@pytest.fixture(scope="module")
def ctx():
    from mulls_b200.registration import Context

    c = Context(0, 4, 300000, 300000)
    yield c
    c.close()


def set_tunables(ctx, **kw):
    for k, v in dict(DEFAULTS, **kw).items():
        ctx.set_tunable(k, v)


def with_params(pair, **kw):
    p = abi.IcpParams.from_buffer_copy(pair["params"])
    for k, v in kw.items():
        setattr(p, k, v)
    return dict(pair, params=p)


def parity_all_drivers(ctx, oracle_mod, pair):
    o, ot = oracle_mod.icp_run(pair["tgt"], pair["src"], pair["params"], pair["init_guess"])
    try:
        for drv in DRIVERS:
            set_tunables(ctx, **drv)
            g, gt = ctx.run_batch([pair], want_trace=True)
            assert_parity(g[0], gt[0], o, ot)
    finally:
        set_tunables(ctx)
    return o, ot


def decoy_pair(small_pair):
    """`small` with the pillar class cut below 500 sources (never shrunk by the duplicate check), plus N_DECOYS pillar
    sources more than 12 m in y from every pillar target, inside the scene's bounding box: a grid sized for
    dis_thre_unit 1.5 (top block reaching at most 12 m along an axis) holds no pillar target for them, but the threshold
    of a growing schedule passes their distance"""
    rng = np.random.default_rng(17)
    tgt = small_pair["tgt"]
    src = [s.copy() for s in small_pair["src"]]
    pil = tgt[abi.PILLAR][:, :3].astype(np.float64)
    lo = np.min([t[:, :3].min(0) for t in tgt if len(t)], axis=0)
    hi = np.max([t[:, :3].max(0) for t in tgt if len(t)], axis=0)
    rows = []
    while len(rows) < N_DECOYS:
        p = np.array([rng.uniform(lo[0] + 5, hi[0] - 5), rng.uniform(pil[:, 1].max() + 12.5, hi[1] - 0.5),
                      rng.uniform(lo[2] + 0.5, hi[2] - 0.5)])
        d = np.abs(pil - p)
        if d.max(1).min() > 12.0 and np.sqrt((d ** 2).sum(1)).min() < 19.0:
            r = src[abi.PILLAR][len(rows)].copy()
            r[:3] = p
            rows.append(r)
    src[abi.PILLAR] = np.concatenate([src[abi.PILLAR][:450], np.array(rows, np.float32)])
    pair = dict(small_pair, src=src)
    return with_params(pair, dis_thre_update_rate=0.8, max_iter_num=14, converge_translation=0.0, converge_rotation_d=0.0)


def test_decoy_pair_is_non_vacuous_on_the_oracle(oracle_mod, small_pair):
    """CPU-side precondition of the decoy test (no GPU): the oracle counts every decoy once the threshold has passed them"""
    pair = decoy_pair(small_pair)
    base = dict(pair, src=[s if c != abi.PILLAR else s[:450] for c, s in enumerate(pair["src"])])
    o, ot = oracle_mod.icp_run(pair["tgt"], pair["src"], pair["params"], pair["init_guess"])
    b, bt = oracle_mod.icp_run(base["tgt"], base["src"], base["params"], base["init_guess"])
    assert o["iters"] == 14
    assert ot["n_corr"][0][abi.PILLAR] == bt["n_corr"][0][abi.PILLAR]  # iteration 0: no decoy within reach
    assert o["n_corr"][abi.PILLAR] - b["n_corr"][abi.PILLAR] == N_DECOYS


@pytest.mark.gpu
def test_decoy_pair_against_the_oracle(ctx, oracle_mod, small_pair):
    """a growing threshold reaches targets far beyond the first iteration's radius: every driver counts them"""
    o, _ = parity_all_drivers(ctx, oracle_mod, decoy_pair(small_pair))
    assert o["n_corr"][abi.PILLAR] >= 450 + N_DECOYS - 5


@pytest.mark.gpu
@pytest.mark.parametrize("sched", [dict(dis_thre_unit=1.5, dis_thre_min=4.0),              # build_pose_graph shape
                                   dict(dis_thre_update_rate=1.0),
                                   dict(dis_thre_update_rate=0.8, converge_translation=0.0, converge_rotation_d=0.0,
                                        max_iter_num=10)],
                         ids=["min_above_unit", "rate1", "rate0.8"])
def test_growing_schedules_against_the_oracle(ctx, oracle_mod, small_pair, sched):
    parity_all_drivers(ctx, oracle_mod, with_params(small_pair, **sched))


# ---- the device's grid through mulls_nn_query ------------------------------------------------------------------------
def rows_of(xyz):
    r = np.zeros((len(xyz), 12), np.float32)
    r[:, :3] = xyz
    r[:, 6] = 1.0
    return r


def brute(tgt, q, chunk=512):
    """argmin under (float32 FLANN distance, index)"""
    t = np.asarray(tgt, np.float32)
    qi, qd = np.empty(len(q), np.int64), np.empty(len(q), np.float32)
    for s in range(0, len(q), chunk):
        d = t[None] - np.asarray(q[s:s + chunk], np.float32)[:, None]
        f = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        qi[s:s + chunk] = np.argmin(f, axis=1)
        qd[s:s + chunk] = f[np.arange(len(f)), qi[s:s + chunk]]
    return qi, qd


def grid_queries(rng, tgt, n=3000):
    """on targets, on the walls of every power-of-two grid anchored at the cloud's minimum (nudged by +-1 ulp),
    jittered, and far outside"""
    t = np.asarray(tgt, np.float32)
    lo, hi = t.min(0), t.max(0)
    k = n // 6
    on = t[rng.integers(0, len(t), k)]
    walls = (lo + (rng.integers(-16, 64, (k, 3)) * np.float32(0.125)).astype(np.float32)).astype(np.float32)
    up, down = np.nextafter(walls, np.float32(np.inf)), np.nextafter(walls, -np.float32(np.inf))
    jit = (t[rng.integers(0, len(t), k)] + rng.normal(0, 0.4, (k, 3))).astype(np.float32)
    far = (rng.uniform(lo - 40, hi + 40, (k, 3))).astype(np.float32)
    return np.concatenate([on, walls, up, down, jit, far]).astype(np.float32)


def geometries():
    rng = np.random.default_rng(41)
    out = {}
    n = 40000  # 1.2 km wide: h0 0.5 at h0_min 0.125
    out["wide_1200m"] = np.c_[rng.uniform(0, 1200, n), rng.uniform(0, 60, n), rng.normal(0, 0.05, n)]
    c2 = synth.make_pair(1001, "c2", n_points=30000)
    out["c2_offset"] = c2["tgt"][abi.GROUND][:, :3].astype(np.float64) + [5000.0, -3000.0, 0.0]
    ax = np.arange(0, 32) * 0.0625
    gx, gy, gz = np.meshgrid(ax, ax, ax[:6], indexing="ij")
    lat = np.stack([gx.ravel(), gy.ravel(), gz.ravel()], 1)
    out["lattice_dup"] = np.concatenate([lat, lat[::7]])  # exact duplicates: ties go to the lower index
    dense = rng.uniform(0, 0.1, (5000, 3)) + 1.0
    out["dense_spot"] = np.concatenate([dense, rng.uniform(-3, 5, (2000, 3))])
    return {k: v.astype(np.float32) for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("tun", [{}, {"leaf_count": 1}, {"leaf_count": 4}, {"hash_slack": 2}, {"h0_min_mm": 250},
                                 {"h0_min_mm": 1000}], ids=["default", "leaf1", "leaf4", "slack2", "h0_250", "h0_1000"])
def test_device_grid_equals_brute_force(ctx, tun):
    rng = np.random.default_rng(42)
    empty = np.zeros((0, 12), np.float32)
    try:
        set_tunables(ctx, **tun)
        for name, xyz in geometries().items():
            tgt = [empty] * 6
            tgt[abi.GROUND] = rows_of(xyz)
            src = [empty] * 6
            src[abi.GROUND] = rows_of(xyz[::50])
            p = abi.default_params()
            p.apply_intersection_filter, p.keep_less_source_points, p.max_iter_num = 0, 0, 1
            p.used_feature_type = b"100000"
            ctx.run_batch([{"tgt": tgt, "src": src, "params": p, "init_guess": np.eye(4)}])
            q = grid_queries(rng, xyz)
            idx, d2 = ctx.nn_query(abi.GROUND, q)
            bi, bd = brute(xyz, q)
            rmax = np.float32(2.5) * np.float32(p.dis_thre_unit)
            inside = bd.astype(np.float64) <= np.float64(rmax) * np.float64(rmax)
            assert inside.sum() > len(q) // 4, name
            bad = np.flatnonzero(inside & ((idx != bi) | (d2 != bd)))
            assert len(bad) == 0, (name, len(bad), q[bad[:3]], idx[bad[:3]], bi[bad[:3]])
            assert np.all(idx[~inside] == -1) and np.all(np.isinf(d2[~inside])), name
    finally:
        set_tunables(ctx)


# ---- pairs with different grids in one batch ----------------------------------------------------------------------------
def wide_pair():
    """a scan pair spread over ~1.1 km (h0 doubled): the small pair's classes tiled along x"""
    base = synth.make_pair(1005, "small")
    tiles = (0.0, 350.0, 700.0, 1050.0)

    def tile(clouds):
        out = []
        for c in clouds:
            parts = []
            for dx in tiles:
                a = c.copy()
                a[:, 0] += np.float32(dx)
                parts.append(a)
            out.append(np.concatenate(parts)[::2].copy())
        return out

    tgt, src = tile(base["tgt"]), tile(base["src"])
    p = abi.IcpParams.from_buffer_copy(base["params"])
    p.target_bound[:] = synth.cloud_bound(tgt)
    return dict(base, tgt=tgt, src=src, params=p)


@pytest.mark.gpu
def test_heterogeneous_batch(ctx, oracle_mod, small_pair):
    """a wide pair, the decoy pair, a normal-shooting pair and `small` in one run_batch: each bit-identical to the
    same pair run alone, and each equal to the oracle"""
    pairs = [wide_pair(), decoy_pair(small_pair), with_params(small_pair, normal_shooting_on=1), small_pair]
    set_tunables(ctx)
    batch, btr = ctx.run_batch(pairs, want_trace=True)
    for k, pair in enumerate(pairs):
        alone, atr = ctx.run_batch([pair], want_trace=True)
        a, b = alone[0], batch[k]
        assert a["code"] == b["code"] and a["iters"] == b["iters"] and a["n_corr"] == b["n_corr"], k
        assert a["n_src"] == b["n_src"], k
        np.testing.assert_array_equal(a["T"], b["T"])
        np.testing.assert_array_equal(a["info"], b["info"])
        np.testing.assert_array_equal(atr[0]["atpa"], btr[k]["atpa"])
        o, ot = oracle_mod.icp_run(pair["tgt"], pair["src"], pair["params"], pair["init_guess"])
        assert_parity(b, btr[k], o, ot)
