"""The per-thread device functions (topay_b200/csrc/*.cuh, TP_HD) instantiated on the CPU by
tests/host_harness.cpp and walked in the kernels' dataflow, against the oracle. Catches maths
errors in the device code without a GPU; the lane mapping itself is covered by the -m gpu tests."""
import numpy as np
import pytest

import host_harness as HH
from topay_b200 import scenes


@pytest.fixture(scope="module")
def harness(oracle, small_scene):
    return HH.Harness(oracle.opt_defaults(), oracle.robot_defaults(), small_scene["desc"], small_scene["field"])


@pytest.fixture(scope="module")
def fields(oracle, small_scene):
    """name -> (oracle field, grid_desc, min_boundary, max_boundary, dims): the default grid with its cuboid scene, and
    the non-square grids A (134 x 80 x 13 @ 0.1) and D (7 x 300 x 5 @ 0.1) of test_gpu_grid_geometry.py with random
    occupancy. On a square grid a transposed stride or an x bound used for y goes unseen."""
    from test_gpu_grid_geometry import grid_spec, random_occupancy
    out = {"default": (small_scene["field"], small_scene["desc"], np.array([-10.0, -10.0, 0.0]),
                       np.array([10.0, 10.0, 1.6]), (200, 200, 16))}
    for name in ("A", "D"):
        desc, lo, hi = grid_spec(name)
        f = oracle.Field(desc)
        f.set_occupancy(*random_occupancy(f.dims, 23))
        f.rebuild()
        out[name] = (f, desc, lo, hi, f.dims)
    return out


def _grid(oracle, fields, name):
    f, desc, lo, hi, dims = fields[name]
    return f, HH.Harness(oracle.opt_defaults(), oracle.robot_defaults(), desc, f), lo, hi, desc.resolution, dims


def test_queries_bit_exact(oracle, small_scene, harness):
    f = small_scene["field"]
    rng = np.random.default_rng(0)
    pos = rng.uniform([-10.5, -10.5, -0.2], [10.5, 10.5, 1.8], (20000, 3))
    _check_queries(f, harness, pos)


@pytest.mark.parametrize("grid", ["A", "D"])
def test_queries_bit_exact_on_other_grids(oracle, fields, grid):
    """test_queries_bit_exact on the non-square grids, over the map +-5 cells in x and y and +-2 cells in z."""
    f, harness, lo, hi, res, _ = _grid(oracle, fields, grid)
    rng = np.random.default_rng(0)
    pos = rng.uniform(lo - [5 * res, 5 * res, 2 * res], hi + [5 * res, 5 * res, 2 * res], (20000, 3))
    _check_queries(f, harness, pos)


def _check_queries(f, harness, pos):
    d0, g0 = f.query3d(pos)
    d1, g1 = harness.query3d(pos)
    assert np.array_equal(d0, d1) and np.array_equal(g0, g1)
    for w in range(3):
        d0, g0 = f.query2d(pos[:, :2], w)
        d1, g1 = harness.query2d(pos[:, :2], w)
        assert np.array_equal(d0, d1) and np.array_equal(g0, g1)


def test_fk_and_linear_time_adjoint(oracle, harness):
    rp = oracle.robot_defaults()
    rng = np.random.default_rng(1)
    for _ in range(100):
        p10 = np.concatenate([rng.uniform(-5, 5, 2), rng.uniform(-3, 3, 1), scenes.random_joints(rng)])
        assert np.abs(oracle.colli_pts(rp, p10)[:, :3] - harness.fk(p10)).max() < 1e-14
        g = rng.normal(size=(12, 3))
        a, b = oracle.colli_grads(rp, p10, g), harness.fk_adjoint(p10, g)
        assert np.abs(a - b).max() <= 1e-13 * np.abs(a).max()


@pytest.mark.parametrize("grid,K", [pytest.param("default", K, id=str(K)) for K in (12, 32, 5)] +
                         [pytest.param("A", K, id=f"A-{K}") for K in (12, 32, 5)])
def test_penalty_dataflow(oracle, fields, grid, K):
    rp, opt = oracle.robot_defaults(), oracle.opt_defaults()
    opt.int_K = K
    f, desc = fields[grid][:2]
    H = HH.Harness(opt, rp, desc, f)
    rng = np.random.default_rng(K)
    # on grid A (13.4 x 8 m) the candidates' 3-8 m spans cross the map's edges
    paths, bv, ba = scenes.short_candidates(3, 11)
    lam, rho = np.array([30.0, -20.0]), np.array([1e4, 2e4])
    for p in paths:
        pr = oracle.prepare_candidate(opt, rp, p, bv[0], ba[0], 64)
        N = pr["piece_num"]
        x = pr["x0"] + 0.05 * rng.normal(size=len(pr["x0"]))
        T = np.array([(0.5 * t + 1) * t + 1 if t > 0 else 1 / ((0.5 * t - 1) * t + 1) for t in x[:N]])
        for stage in (1, 2):
            coeff = oracle.eval_one(opt, rp, f, stage, N, pr["head_pva"], pr["tail_pva"], pr["start_xy"],
                                    pr["end_xy"], pr["init_inner_xy"][:N], lam, rho, x)[3]
            _, gdC, gdT, tm, fx0 = oracle.penalty_only(opt, rp, f, stage, N, coeff, T, pr["start_xy"], pr["end_xy"],
                                                       pr["init_inner_xy"][:N], lam, rho)
            gdC1, gdT1, tm1, fx1 = H.penalty_eval(stage, N, coeff, T, pr["start_xy"], pr["end_xy"],
                                                  pr["init_inner_xy"][:N], lam, rho)
            assert np.abs(gdC - gdC1).max() <= 1e-12 * np.abs(gdC).max()
            assert np.abs(gdT - gdT1).max() <= 1e-12 * np.abs(gdT).max()
            assert np.abs(tm - tm1).max() <= 1e-12 * np.abs(tm).max()
            assert np.abs(fx0 - fx1).max() < 1e-13


def test_rog_lookups_bit_exact(oracle):
    """rog_query.cuh (ring hash, six query kinds, isLineFree2d walk, the solver's field-kind dispatch) on the
    CPU against the oracle's ROG field: same buffers, bit-identical answers, wrapped positions included."""
    from topay_b200._structs import rog_desc
    desc = rog_desc(half_prob_map_size_i=(30, 22, 9), prob_resolution=0.1, esdf_resolution=0.1,
                    local_update_box=(5.0, 3.0, 1.5), map_sliding_en=True)
    orc = oracle.RogField(desc)
    rng = np.random.default_rng(4)
    odom = (0.43, -0.31, 0.12)
    orc.slide(odom)
    hits = np.array(odom) + rng.uniform(-1, 1, (500, 3)) * np.array([2.8, 2.0, 0.8])
    orc.update_counters(hits, np.full(500, 1), np.full(500, 3))
    orc.update_esdf(odom)
    H = HH.RogHarness(orc)
    pos = np.concatenate([np.array(odom) + rng.uniform(-1, 1, (4000, 3)) * np.array([2.0, 1.3, 0.6]),
                          rng.uniform(-40, 40, (500, 3))])
    for kind in range(6):
        d0, g0 = orc.query(kind, pos)
        d1, g1 = H.query(kind, pos)
        assert np.array_equal(d0, d1), kind
        if kind < 3:
            assert np.array_equal(g0, g1), kind
    s = (np.array(odom) + rng.uniform(-1, 1, (3000, 3)) * np.array([2.0, 1.3, 0.0]))[:, :2]
    e = (np.array(odom) + rng.uniform(-1, 1, (3000, 3)) * np.array([2.0, 1.3, 0.0]))[:, :2]
    for thr in (0.0, 0.15, 0.4):
        assert np.array_equal(H.line_free(s, e, thr), orc.is_line_free2d(s, e, thr)), thr
    # the dispatch GridMap's use_rog branches go through (grid_map.h:256-267, 307-322, 364-392, 443-461)
    d2, g2, d3, g3, v2, v3 = H.dispatch(pos)
    p0 = pos.copy()
    p0[:, 2] = 0.0
    e2, eg2 = orc.query(1, p0)
    e3, eg3 = orc.query(0, pos)
    assert np.array_equal(d2, e2) and np.array_equal(g2, eg2[:, :2]) and np.array_equal(v2, e2)
    assert np.array_equal(d3, e3) and np.array_equal(g3, eg3) and np.array_equal(v3, e3)


def test_field_predicates_bit_exact(oracle, small_scene, harness):
    f = small_scene["field"]
    rng = np.random.default_rng(8)
    n = 5000
    p2, q2 = rng.uniform(-10.3, 10.3, (n, 2)), rng.uniform(-10.3, 10.3, (n, 2))
    p3 = np.concatenate([rng.uniform(-10.3, 10.3, (n, 2)), rng.uniform(-0.2, 1.8, (n, 1))], axis=1)
    idx = rng.integers(-5, 206, (n, 2))
    _check_predicates(f, harness, p2, q2, p3, idx)


@pytest.mark.parametrize("grid", ["A", "D"])
def test_field_predicates_bit_exact_on_other_grids(oracle, fields, grid):
    """test_field_predicates_bit_exact on the non-square grids: positions over the map +-3 cells (z +-2 cells), cell
    indices -5 .. max(dims) + 5 on both axes."""
    f, harness, lo, hi, res, dims = _grid(oracle, fields, grid)
    rng = np.random.default_rng(8)
    n = 5000
    p2, q2 = rng.uniform(lo[:2] - 3 * res, hi[:2] + 3 * res, (n, 2)), rng.uniform(lo[:2] - 3 * res, hi[:2] + 3 * res, (n, 2))
    p3 = np.concatenate([rng.uniform(lo[:2] - 3 * res, hi[:2] + 3 * res, (n, 2)),
                         rng.uniform(lo[2] - 2 * res, hi[2] + 2 * res, (n, 1))], axis=1)
    idx = rng.integers(-5, max(dims) + 6, (n, 2))
    _check_predicates(f, harness, p2, q2, p3, idx)


def _check_predicates(f, harness, p2, q2, p3, idx):
    for thr, crit in ((0.0, False), (0.3, True)):
        c2, c3, line, cd, ci = HH.field_misc(harness, p2, q2, p3, idx, thr, crit)
        assert np.array_equal(c2, f.is_collision(p2, thr)) and np.array_equal(c3, f.is_collision(p3, thr))
        assert np.array_equal(line, f.line_collision2d(p2, q2, thr))
        assert np.array_equal(cd, f.dist_coarse2d(p2, crit)) and np.array_equal(ci, f.dist_coarse2i(idx, crit))


def test_line_visibility_ray_bit_exact(oracle, small_scene, harness):
    """N2: tp_line_visib (field_query.cuh; TopologyPRM::lineVisib over the planner's RayCaster) instantiated on the CPU
    against the oracle: verdicts and blocking points of segments across the scene, ends outside the map, degenerate rays."""
    f = small_scene["field"]
    rng = np.random.default_rng(9)
    n = 6000
    p1 = np.concatenate([rng.uniform(-9.8, 9.8, (n, 2)), np.zeros((n, 1))], axis=1)
    p2 = p1 + np.concatenate([rng.normal(size=(n, 2)) * rng.choice([0.05, 0.5, 4.0], (n, 1)), np.zeros((n, 1))], axis=1)
    p2[::40] = p1[::40]
    p2[1::40, :2] *= 1.3
    for thr, crit in ((0.0, False), (0.25, True)):
        va, pa = harness.line_visib(p1, p2, thr, crit)
        vb, pb = f.line_visib(p1, p2, thr, crit)
        assert np.array_equal(va, vb) and np.array_equal(pa[~va], pb[~vb]) and np.isnan(pa[va]).all()


def test_traj_evaluation_bit_exact(oracle):
    """traj.cuh (locatePieceIdx, Piece::getPos/getVel/getAcc, MomaTraj::getState/getDState) on the CPU against
    the oracle, fed with the oracle's pose table."""
    rng = np.random.default_rng(12)
    N = 5
    T = rng.uniform(0.6, 1.8, N)
    coeff = rng.normal(size=(6 * N, 9)) * (0.5 ** np.tile(np.arange(6), N))[:, None]
    tr = (T, coeff, np.array([0.3, -0.2, 0.7]))
    seq = oracle.traj_car_seq([tr])[0]
    t = np.concatenate([np.linspace(-0.3, T.sum() + 0.3, 301), np.cumsum(T), [0.0, T.sum()]])
    st, ds, pva = HH.traj_sample(T, coeff, seq, t)
    est, eds = oracle.traj_sample([tr], t[None])
    assert np.array_equal(ds, eds[0])
    # the state adds one Simpson step with sin/cos: same libm on both sides here
    assert np.abs(st - est[0]).max() <= 1e-15 * max(1.0, np.abs(est[0]).max())


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 16, 17, 32, 33, 34, 64, 65, 80, 83, 200, 513, 800, 803])
def test_edt_line_divide_and_conquer(n):
    """a20: the per-line arithmetic of the strided EDT passes (edt_line.cuh) in the kernel's schedule (skip distances, chunk boundaries, halving inside the chunks) against the
    brute-force minimum  min_v (q - v)^2 + f(v)  of both transforms: dense, sparse, single-source, all-source and
    source-free lines, first-pass (squared int16) and second-pass (arbitrary squared distances) value ranges."""
    import host_harness as hh
    INF = 1 << 29
    rng = np.random.default_rng(n)
    q = np.arange(n)
    d2 = (q[:, None] - q[None, :]) ** 2
    cases = []
    for density in (0.0, 0.003, 0.02, 0.3, 0.9, 1.0):
        occ = rng.random(n) < density
        # second-pass style input: occupied cells are sources of the positive transform (0) and carry their
        # negative value; free cells carry a positive value (or INF)
        pos = np.where(occ, 0, np.where(rng.random(n) < 0.5, rng.integers(1, 90, n) ** 2 + rng.integers(0, 50, n), INF))
        neg = np.where(occ, np.where(rng.random(n) < 0.9, rng.integers(1, 6, n) ** 2, INF), 0)
        cases.append((pos, neg))
    one = np.full(n, INF)
    one[n // 3] = 7
    cases.append((one, np.zeros(n, dtype=np.int64)))
    for pos, neg in cases:
        packed = np.where(neg > 0, -neg, pos).astype(np.int32)
        assert not (packed == 0).any() or n >= 1
        packed[packed == 0] = INF          # a free cell with no finite value
        fp, fn = np.maximum(packed, 0).astype(np.int64), np.maximum(-packed.astype(np.int64), 0)
        exp_p, exp_n = (d2 + fp[None, :]).min(axis=1), (d2 + fn[None, :]).min(axis=1)
        for chunk in (4, 8, 32):
            got_p, got_n = hh.edt_line(packed, chunk)
            assert np.array_equal(got_p, np.minimum(exp_p, INF)) and np.array_equal(got_n, exp_n), chunk
        # the two-scan lower envelope (thread per line on large grids) answers the same line
        for segments in (1, 4):
            got_p, got_n, depth = hh.edt_scan_line(packed, segments)
            assert np.array_equal(got_p, np.minimum(exp_p, INF)) and np.array_equal(got_n, np.minimum(exp_n, INF))
            assert depth <= max(32, (n + segments - 1) // segments + 31)
    assert hh.lib().hh_sq16(-16383) == -INF and hh.lib().hh_sq16(16383) == INF and hh.lib().hh_sq16(-5) == -25
