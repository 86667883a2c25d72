"""GPU parity gates, all through the C ABI (topay_b200/libtopay_b200.so):

* field: integer squared-distance grids and fp64 ESDF grids bit-exact against the oracle and the
  golden fixture, incl. empty / full / ragged grids and the accumulate-critical quirk;
* queries: value and gradient against the oracle (<= 1e-12 absolute; FMA contraction only);
* one cost/gradient evaluation: <= 1e-9 relative (north_star tolerance) on cost, 13 term costs,
  gradient and spline coefficients, both stages, K in {1, 2, 3, 4, 5, 8, 12, 16, 31, 32}, ragged piece counts in a
  batch, candidates of 33..64 pieces;
* batched solve: identical line-search decisions and f within 1e-9 over the first accepted
  iterations; final cost / duration inside the reference algorithm's own sensitivity band
  (DESIGN.md "final-trajectory tolerance"); end-point constraint met; selection rule. Also in timed mode, whose
  plain launches always split k_cand into its three halves: bit-identical to the graph-mode solve.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INT_MAX = np.iinfo(np.int32).max


@pytest.fixture(scope="module")
def gpu_scene(small_scene):
    import topay_b200 as tp
    gm = tp.GridMap(small_scene["desc"], device=0)
    gm.regenerateMap(small_scene["points"])
    return gm


def _compare_fields(gm, of):
    for which in (0, 1, 2, 3):
        a, b = gm.getSqDist(which), of.download_sqdist(which)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), f"integer grid {which}"
        assert np.array_equal(gm._download(which), of.download(which)), f"esdf {which}"


def test_field_bit_exact_default_grid(gpu_scene, small_scene):
    of = small_scene["field"]
    _compare_fields(gpu_scene, of)
    assert np.array_equal(gpu_scene.getOccBuffer3d(), of.download_occupancy(3))
    assert np.array_equal(gpu_scene.getOccBuffer2d(), of.download_occupancy(0))
    assert np.array_equal(gpu_scene.getOccBuffer2dCritical(), of.download_occupancy(2))


def test_field_golden_fixture():
    import topay_b200 as tp
    z = np.load(os.path.join(G, "field_small.npz"))
    gm = tp.GridMap(tp.grid_desc(map_size=tuple(z["map_size"]), resolution=float(z["resolution"])))
    gm.loadMap(z["occ_2d"], z["occ_3d"], z["occ_2d_critical"])
    sqp, sqn = gm.getSqDist(3)
    assert np.array_equal(sqp, z["sq_pos_3d"]) and np.array_equal(sqn, z["sq_neg_3d"])
    assert np.array_equal(gm.getESDFBuffer3d(), z["esdf_3d"])
    assert np.array_equal(gm.getESDFBuffer2d(), z["esdf_2d"])
    assert np.array_equal(gm.getESDFBuffer2dInflate(), z["esdf_2d_inflate"])
    assert np.array_equal(gm.getESDFBuffer2dCritical(), z["esdf_2d_critical"])
    d, g = gm.getDisWithGradI3d(z["query_pos"])
    assert np.abs(d - z["query_d3"]).max() <= 1e-12 and np.abs(g - z["query_g3"]).max() <= 1e-11


@pytest.mark.parametrize("shape,fill", [((13, 10, 6), 0.05), ((37, 19, 3), 0.3), ((5, 70, 33), 0.9),
                                        ((6, 5, 4), 0.0), ((6, 5, 4), 1.0), ((1, 1, 1), 1.0)])
def test_field_ragged_and_degenerate(oracle, shape, fill):
    import topay_b200 as tp
    res = 0.1
    desc = tp.grid_desc(map_size=tuple((s - 0.5) * res for s in shape), resolution=res)
    gm, of = tp.GridMap(desc), oracle.Field(desc)
    assert gm.voxel_num == shape == of.dims
    rng = np.random.default_rng(sum(shape))
    occ3 = (rng.random(shape) < fill).astype(np.int8)
    occ2 = (rng.random(shape[:2]) < fill).astype(np.int8)
    occ2c = (rng.random(shape[:2]) < fill).astype(np.int8)
    gm.loadMap(occ2, occ3, occ2c)
    of.set_occupancy(occ3, occ2, occ2c)
    of.rebuild()
    _compare_fields(gm, of)
    if fill == 0.0:
        assert (gm.getSqDist(3)[0] == INT_MAX).all()


@pytest.mark.parametrize("shape,fill", [((13, 10, 16), 0.05), ((37, 19, 32), 0.3), ((5, 70, 48), 0.9), ((40, 3, 128), 0.5),
                                        ((21, 300, 80), 0.002), ((260, 9, 64), 0.6), ((6, 5, 4), 0.0), ((6, 5, 4), 1.0),
                                        ((3, 2, 16), 0.0), ((3, 2, 16), 1.0), ((1, 1, 1), 1.0)])
def test_field_thread_per_line_kernels(oracle, shape, fill, monkeypatch):
    """a20: the kernels large grids take (one thread per line: k_edt_contig_thread for z lines of 16 NV cells, the two-scan
    lower envelope k_edt_scan for the strided passes and the 2-D maps), forced onto small ragged / empty / full grids:
    bit-identical to the oracle, and to the kernels small grids take."""
    import topay_b200 as tp
    res = 0.1
    desc = tp.grid_desc(map_size=tuple((s - 0.5) * res for s in shape), resolution=res)
    of = oracle.Field(desc)
    rng = np.random.default_rng(sum(shape) + 1)
    occ3 = (rng.random(shape) < fill).astype(np.int8)
    occ2 = (rng.random(shape[:2]) < fill).astype(np.int8)
    occ2c = (rng.random(shape[:2]) < fill).astype(np.int8)
    of.set_occupancy(occ3, occ2, occ2c)
    of.rebuild()
    got = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("TOPAY_EDT_SCAN", mode)
        gm = tp.GridMap(desc)
        gm.loadMap(occ2, occ3, occ2c)
        _compare_fields(gm, of)
        got[mode] = gm._download(3)
        gm.close()
    assert np.array_equal(got["0"], got["1"])


def test_rasterize_and_critical_quirk(oracle, small_scene):
    import topay_b200 as tp
    from topay_b200 import scenes
    gm, of = tp.GridMap(small_scene["desc"]), oracle.Field(small_scene["desc"])
    for seed in (1, 2):      # second scene: occ_2d / occ_3d reset, critical occupancy accumulates
        pts, _ = scenes.tables_scene(seed) if seed == 1 else scenes.cuboids_scene(seed)
        gm.regenerateMap(pts)
        of.clear(False)
        of.rasterize(pts)
        of.rebuild()
        assert np.array_equal(gm.getOccBuffer3d(), of.download_occupancy(3))
        assert np.array_equal(gm.getOccBuffer2dCritical(), of.download_occupancy(2))
        _compare_fields(gm, of)
    gm.rasterize(np.zeros((0, 3), np.float32))      # empty cloud is a no-op


def test_queries_and_collision(gpu_scene, small_scene, oracle):
    of = small_scene["field"]
    rng = np.random.default_rng(1)
    pos = rng.uniform([-10.5, -10.5, -0.2], [10.5, 10.5, 1.8], (50000, 3))
    d0, g0 = of.query3d(pos)
    d1, g1 = gpu_scene.getDisWithGradI3d(pos)
    assert np.abs(d0 - d1).max() <= 1e-12 and np.abs(g0 - g1).max() <= 1e-11
    v0, v1 = of.distance3d(pos), gpu_scene.getDistance3d(pos)
    assert np.array_equal(v0 == 1e10, v1 == 1e10) and np.abs(v0 - v1).max() <= 1e-12
    for w, kw in ((0, {}), (1, dict(inflate=True)), (2, dict(critical=True))):
        d0, g0 = of.query2d(pos[:, :2], w)
        d1, g1 = gpu_scene.getDisWithGradI2d(pos[:, :2], **kw)
        assert np.abs(d0 - d1).max() <= 1e-12 and np.abs(g0 - g1).max() <= 1e-11
    assert np.abs(of.distance2d(pos[:, :2]) - gpu_scene.getDistance2d(pos[:, :2])).max() <= 1e-12
    from topay_b200 import scenes
    rp = oracle.robot_defaults()
    states = np.concatenate([rng.uniform(-9, 9, (4000, 2)), rng.uniform(-3, 3, (4000, 1)),
                             np.stack([scenes.random_joints(rng) * 1.02 for _ in range(4000)])], axis=1)
    a = of.whole_body_collision(rp, states).astype(bool)
    b = gpu_scene.isWholeBodyCollision(states)
    assert (a != b).mean() < 1e-3 and 0.05 < a.mean() < 0.999    # only threshold-grazing states may differ
    with pytest.raises(Exception):
        import topay_b200 as tp
        tp.GridMap(small_scene["desc"]).getDisWithGradI3d(pos[:4])    # not built yet -> NOT_READY


def _eval_batch(solver, stage, prep, xs, lam, rho):
    return solver.evaluate(stage, [q["piece_num"] for q in prep], [q["head_pva"] for q in prep],
                           [q["tail_pva"] for q in prep], [q["start_xy"] for q in prep], [q["end_xy"] for q in prep],
                           [q["init_inner_xy"] for q in prep], xs, lam, rho)


def _check_eval_against_oracle(solver, of, oracle, opt, rp, prep, seed):
    """One evaluation of every candidate of `prep`, both stages, against the oracle; returns the worst relative
    deviation."""
    import topay_b200 as tp
    n_c = len(prep)
    rng = np.random.default_rng(seed)
    xs = [q["x0"] + 0.05 * rng.normal(size=len(q["x0"])) for q in prep]
    lam, rho = np.tile([30.0, -20.0], (n_c, 1)), np.tile([1e4, 2e4], (n_c, 1))
    worst = 0.0
    for stage in (1, 2):
        ev = _eval_batch(solver, stage, prep, xs, lam, rho)
        for c, q in enumerate(prep):
            N = q["piece_num"]
            f, g, terms, coeff, fxy = oracle.eval_one(opt, rp, of, stage, N, q["head_pva"], q["tail_pva"],
                                                      q["start_xy"], q["end_xy"], q["init_inner_xy"][:N], lam[c],
                                                      rho[c], xs[c])
            n = tp.num_vars(N)
            e = [np.abs(ev["coeff"][c, :6 * N] - coeff).max() / np.abs(coeff).max(), abs(ev["cost"][c] - f) / abs(f),
                 np.abs(ev["terms"][c] - terms).max() / np.abs(terms).max(),
                 np.abs(ev["grad"][c, :n] - g).max() / np.abs(g).max()]
            worst = max(worst, *e)
            assert e[0] <= 1e-10 and e[1] <= 1e-9 and e[2] <= 1e-9 and e[3] <= 1e-9, (stage, c, e)
            assert np.abs(ev["final_xy"][c] - fxy).max() <= 1e-12
    return worst


# K-hat = 4 (K 1..4: eight pieces per warp, 16 values per lane in the transpose-reduce, lane K-hat - 1 owns gdT),
# K-hat = 8 with and without end-node warps (8, 5), K-hat = 16 (12, 16), K-hat = 32 with and without them (32, 31)
@pytest.mark.parametrize("K", [12, 32, 5, 16, 1, 2, 3, 4, 8, 31])
def test_eval_parity(gpu_scene, small_scene, oracle, K):
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K = K
    paths, bv, ba = scenes.short_candidates(6, 100 + K)      # ragged: 3..10 pieces in one batch
    prep = [tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 16) for p in paths]
    assert len({q["piece_num"] for q in prep}) > 1
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=8, max_pieces=16, opt_param=opt, robot=rp)
    worst = _check_eval_against_oracle(solver, small_scene["field"], oracle, opt, rp, prep, K)
    print(f"K={K}: worst relative deviation from the oracle {worst:.2e}")


@pytest.mark.parametrize("K", [4, 16, 31, 32])
def test_eval_parity_long_candidates(gpu_scene, small_scene, oracle, K):
    """Long candidates in one ragged batch (33, 40 and 64 pieces at max_pieces = 64), both stages: more than 32 pieces
    put the end nodes of K = K-hat on two warps, K-hat = 4 runs 8 piece groups per candidate, and stage 1 runs at
    64 pieces, which the short candidates above never reach."""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K, opt.sample_interval = K, 1e9
    paths, bv, ba = scenes.synthetic_batch(3, 1234 + K)
    prep = []
    for p, pieces in zip(paths, (33, 40, 64)):
        opt.min_piece_num = pieces
        prep.append(tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 64))
    assert [q["piece_num"] for q in prep] == [33, 40, 64]
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=3, max_pieces=64, opt_param=opt, robot=rp)
    worst = _check_eval_against_oracle(solver, small_scene["field"], oracle, opt, rp, prep, K)
    print(f"K={K}, 33..64 pieces: worst relative deviation from the oracle {worst:.2e}")


def test_eval_golden_and_full_size(gpu_scene, small_scene, oracle):
    import topay_b200 as tp
    from topay_b200 import scenes
    z = np.load(os.path.join(G, "eval_cases.npz"))
    rp = tp.robot_params_default()
    for c in range(int(z["n_cases"])):
        k = f"c{c}"
        opt = tp.opt_params_default()
        opt.int_K, opt.min_piece_num = int(z[f"{k}_K"]), int(z[f"{k}_min_pieces"])
        pr = tp.prepare_candidate(opt, rp, z[f"{k}_path"], np.zeros((10, 2)), np.zeros((10, 2)), 16)
        solver = tp.MomaTrajOpt(gpu_scene, max_cand=1, max_pieces=16, opt_param=opt, robot=rp)
        ev = _eval_batch(solver, int(z[f"{k}_stage"]), [pr], [z[f"{k}_x"]], z[f"{k}_lambda"][None], z[f"{k}_rho"][None])
        n = len(z[f"{k}_x"])
        assert abs(ev["cost"][0] - float(z[f"{k}_cost"])) <= 1e-9 * abs(float(z[f"{k}_cost"]))
        assert np.abs(ev["grad"][0, :n] - z[f"{k}_grad"]).max() <= 1e-9 * np.abs(z[f"{k}_grad"]).max()
        solver.close()
    # BASELINE size (64 pieces x K = 32): one candidate against the oracle + linearity of the ALM term
    opt = tp.opt_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    paths, bv, ba = scenes.synthetic_batch(3, 1234)
    prep = [tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 64) for p in paths]
    assert all(q["piece_num"] == 64 for q in prep)
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=3, max_pieces=64, opt_param=opt, robot=rp)
    xs = [q["x0"] for q in prep]
    lam, rho = np.zeros((3, 2)), np.full((3, 2), 1e4)
    ev = _eval_batch(solver, 2, prep, xs, lam, rho)
    q = prep[0]
    f, g, terms, coeff, fxy = oracle.eval_one(opt, rp, small_scene["field"], 2, 64, q["head_pva"], q["tail_pva"],
                                              q["start_xy"], q["end_xy"], q["init_inner_xy"], lam[0], rho[0], xs[0])
    assert abs(ev["cost"][0] - f) <= 1e-9 * abs(f) and np.abs(ev["grad"][0] - g).max() <= 1e-9 * np.abs(g).max()
    # size-independent property: the cost is affine in lambda at fixed x, with slope final_xy
    ev2 = _eval_batch(solver, 2, prep, xs, lam + 5.0, rho)
    slope = (ev2["cost"] - ev["cost"]) / 5.0
    assert np.abs(slope - ev["final_xy"].sum(axis=1) - 0.5 * 5.0 * (2.0 / 1e4)).max() <= 1e-6 * (1 + np.abs(slope).max())


RESULT_KEYS = ("status", "lbfgs_code", "evals", "iters", "alm_rounds", "cost", "T", "coeff", "x", "final_xy_err")


def test_solve_trace_and_band(gpu_scene, small_scene, oracle):
    _solve_trace_and_band(gpu_scene, small_scene, oracle, timed=False)


def test_solve_trace_and_band_timed(gpu_scene, small_scene, oracle):
    """Timed mode: per-launch CUDA events and plain launches, which always run k_cand as three launches (adjoint,
    L-BFGS, generate) handing their state over through global memory; graph mode runs this pool as one fused launch.
    Both must replay the oracle, and the timed solve must equal the graph-mode one bit for bit."""
    _solve_trace_and_band(gpu_scene, small_scene, oracle, timed=True)


def _solve_trace_and_band(gpu_scene, small_scene, oracle, timed):
    import topay_b200 as tp
    z = np.load(os.path.join(G, "solve_cases.npz"))
    n = int(z["n"])
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths = [z[f"s{c}_path"] for c in range(n)]
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=n, max_pieces=16, opt_param=opt, robot=rp)
    solver.set_trace(4000)
    res = solver.optimizeTrajBatch(paths, np.zeros((n, 10, 2)), np.zeros((n, 10, 2)))
    if timed:
        graph = res
        graph_trace = [solver.trace(c) for c in range(n)]
        solver.set_timed(True)
        res = solver.optimizeTrajBatch(paths, np.zeros((n, 10, 2)), np.zeros((n, 10, 2)))
        st = solver.stats()
        # one lane; every batch split: k_list_roll + 16 ticks x (3 evaluation kernels + 3 halves of k_cand)
        assert st["eval_launches"] == st["ticks"] and st["kernel_launches"] == 2 + 97 * st["ticks"] // 16, st
        for k in RESULT_KEYS:
            assert np.array_equal(res[k], graph[k]), k
        for c in range(n):
            assert np.array_equal(solver.trace(c), graph_trace[c]), c
    for c in range(n):
        assert res["status"][c] == int(z[f"s{c}_status"]) == 1
        assert res["piece_num"][c] == int(z[f"s{c}_piece_num"])
        # the first accepted iterations replay the oracle's: same k, same number of line-search
        # evaluations, same step, f within 1e-9 relative
        tg, tc = solver.trace(c), z[f"s{c}_trace"]
        m = 8
        assert np.array_equal(tg[:m, 2:], tc[:m, 2:]) and np.allclose(tg[:m, 1], tc[:m, 1], rtol=1e-9, atol=0)
        assert np.abs(tg[:m, 0] - tc[:m, 0]).max() <= 1e-9 * np.abs(tc[:m, 0]).max()
        # final trajectory: inside the reference algorithm's own +-1e-15-perturbation band, widened 3x
        lo, hi = z[f"s{c}_cost_band"]
        w = max(hi - lo, 0.02 * hi)
        assert lo - 3 * w <= res["cost"][c] <= hi + 3 * w, (c, res["cost"][c], lo, hi)
        lo, hi = z[f"s{c}_duration_band"]
        w = max(hi - lo, 0.02 * hi)
        assert lo - 3 * w <= res["duration"][c] <= hi + 3 * w
        assert np.linalg.norm(res["final_xy_err"][c]) < opt.alm_tolerance
        assert abs(res["T"][c, :res["piece_num"][c]].sum() - res["duration"][c]) < 1e-9
        # length of the base path and clearances (north-star: "cost, length and clearance"), all computed on
        # the device from the device's own trajectory, against the same kind of band
        tr = solver.getTraj(c)
        seq = tr.car_seq
        xy = np.concatenate([seq[:, :2], tr.getState(tr.getTotalDuration())[None, :2]])
        length = np.linalg.norm(np.diff(xy, axis=0), axis=1).sum()
        solver.checkFeasible(tr)
        radii = np.array([rp.colli_point_radius[i] for i in range(16) if rp.colli_points[i] != 0.0])
        clear_base = solver.constraints["min_dist"][0]
        clear_arm = (solver.constraints["min_dist_mani"][0, :len(radii)] - radii).min()
        for val, key, floor in ((length, "length", 0.02 * length), (clear_base, "clear_base", 0.05),
                                (clear_arm, "clear_arm", 0.05)):
            lo, hi = z[f"s{c}_{key}_band"]
            w = max(hi - lo, floor)
            assert lo - 3 * w <= val <= hi + 3 * w, (c, key, val, lo, hi)
    ok = np.nonzero(res["status"] == 1)[0]
    assert res["best_by_duration"] == ok[np.argmin(res["duration"][ok])]
    assert res["best_by_cost"] == ok[np.argmin(res["cost"][ok])]
    # reference call shape: one candidate, bool result, traj_cost, getTraj
    one = tp.MomaTrajOpt(gpu_scene, max_cand=1, max_pieces=16, opt_param=opt, robot=rp)
    assert one.optimizeTraj(paths[0], np.zeros((10, 2)), np.zeros((10, 2))) is True
    traj = one.getTraj()
    assert traj.is_init and abs(traj.getTotalDuration() - res["duration"][0]) < 1e-6 * res["duration"][0]
    assert abs(one.traj_cost - res["cost"][0]) <= 1e-9 * abs(res["cost"][0])      # deterministic re-run


def test_capacity_errors(gpu_scene):
    import topay_b200 as tp
    from topay_b200 import _lib, scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=2, max_pieces=4, opt_param=opt, robot=rp)
    paths, bv, ba = scenes.short_candidates(3, 7)
    with pytest.raises(_lib.TopayError) as e:
        solver.optimizeTrajBatch(paths, bv, ba)              # 3 candidates > max_cand
    assert e.value.code == _lib.ERR_TOO_LARGE
    long_paths, bv2, ba2 = scenes.synthetic_batch(1, 3)
    with pytest.raises(_lib.TopayError):
        solver.optimizeTrajBatch(long_paths, bv2, ba2)       # needs more pieces than max_pieces
    opt.int_K = 64
    with pytest.raises(_lib.TopayError):
        tp.MomaTrajOpt(gpu_scene, max_cand=1, max_pieces=4, opt_param=opt, robot=rp)


def test_baseline_size_field_properties(oracle):
    """800 x 800 x 80 @ 0.05 m (BASELINE configs[3]): properties that do not need the oracle at full
    size + exact agreement with brute force at random voxels."""
    import topay_b200 as tp
    from topay_b200 import scenes
    desc = tp.grid_desc(map_size=(40.0, 40.0, 4.0), resolution=0.05)
    gm = tp.GridMap(desc)
    assert gm.voxel_num == (800, 800, 80)
    pts, _ = scenes.cuboids_scene(7, size_x=40.0, size_y=40.0, scale=2.0)
    gm.regenerateMap(pts)
    occ = gm.getOccBuffer3d()
    sqp, sqn = gm.getSqDist(3)
    assert (sqp[occ == 1] == 0).all() and (sqn[occ == 0] == 0).all() and (sqp[occ == 0] > 0).all()
    # squared EDT of neighbours: |sqrt(a) - sqrt(b)| <= 1 along every axis
    r = np.sqrt(sqp.astype(np.float64))
    for ax in range(3):
        assert np.abs(np.diff(r, axis=ax)).max() <= 1.0 + 1e-12
    src = np.argwhere(occ == 1)
    rng = np.random.default_rng(0)
    for p in rng.integers(0, [800, 800, 80], (40, 3)):
        assert sqp[tuple(p)] == ((src - p) ** 2).sum(1).min()
    e = gm.getESDFBuffer3d()
    dp, dn = 0.05 * np.sqrt(sqp.astype(np.float64)), 0.05 * np.sqrt(sqn.astype(np.float64))
    assert np.array_equal(e, np.where(dn > 0, dp + (-dn + 0.05), dp))
    gm.updateESDF()                                              # idempotent
    assert np.array_equal(gm.getESDFBuffer3d(), e)
    print("800x800x80 rebuild ms (total, 3-D part):", gm.last_rebuild_ms())


def test_front_end_predicates_and_coarse_lookups(gpu_scene, small_scene):
    """isCollision2d/3d, isLineCollisionGrid2d, getDistCoarse2d/2i (grid_map.h:511-611, 695-724, 887-940):
    exact against the oracle except where an interpolated distance sits within 1e-12 of the threshold."""
    of = small_scene["field"]
    rng = np.random.default_rng(8)
    p2 = rng.uniform(-10.3, 10.3, (20000, 2))
    p3 = np.concatenate([rng.uniform(-10.3, 10.3, (20000, 2)), rng.uniform(-0.2, 1.8, (20000, 1))], axis=1)
    for thr in (0.0, 0.25, 0.4):
        for pos, got in ((p2, gpu_scene.isCollision2d(p2, thr)), (p3, gpu_scene.isCollision3d(p3, thr))):
            exp = of.is_collision(pos, thr)
            d = of.distance2d(pos) if pos.shape[1] == 2 else of.distance3d(pos)
            near = np.abs(d - thr) < 1e-12
            assert np.array_equal(got[~near], exp[~near]) and 0 < exp.sum() < len(exp)
    a, b = rng.uniform(-9.9, 9.9, (5000, 2)), rng.uniform(-9.9, 9.9, (5000, 2))
    b[:50] = a[:50]
    b[50:100] = rng.uniform(-12, 12, (50, 2))          # leaves the map
    for thr in (0.0, 0.3):
        got, exp = gpu_scene.isLineCollisionGrid2d(a, b, thr), of.line_collision2d(a, b, thr)
        assert np.array_equal(got, exp) and 0 < exp.sum() < len(exp)
    for crit in (False, True):
        assert np.array_equal(gpu_scene.getDistCoarse2d(p2, crit), of.dist_coarse2d(p2, crit))
        idx = rng.integers(-5, 206, (5000, 2))
        assert np.array_equal(gpu_scene.getDistCoarse2i(idx, crit), of.dist_coarse2i(idx, crit))


def test_line_visibility_rays(gpu_scene, small_scene):
    """N2: TopologyPRM::lineVisib on the device (topay_field_line_visible) — verdict and blocking point of 20 000
    segments (long, short, degenerate, leaving the map) against the oracle (= the reference's lineVisib over its own
    RayCaster, test_ref_pin.py::test_line_visib_bit_exact), inflated and critical map: bit-identical."""
    of = small_scene["field"]
    rng = np.random.default_rng(21)
    n = 20000
    p1 = np.concatenate([rng.uniform(-9.8, 9.8, (n, 2)), np.zeros((n, 1))], axis=1)
    p2 = p1 + np.concatenate([rng.normal(size=(n, 2)) * rng.choice([0.05, 0.5, 4.0], (n, 1)), np.zeros((n, 1))], axis=1)
    p2[::40] = p1[::40]
    p2[1::40, :2] *= 1.3          # some ends outside the map (cells clamped by getDistCoarse2i)
    for crit in (False, True):
        for thresh in (0.0, 0.25):
            vg, pg = gpu_scene.lineVisib(p1, p2, thresh, crit)
            vo, po = of.line_visib(p1, p2, thresh, crit)
            assert np.array_equal(vg, vo)
            assert np.array_equal(pg[~vg], po[~vo])
            assert np.isnan(pg[vg]).all()
    assert 0.05 < vg.mean() < 0.98


def test_same_topo_paths_batch(gpu_scene, small_scene):
    """N2: TopologyPRM::sameTopoPath for all pairs of a set of paths in one launch (topay_field_same_topo_paths:
    host discretizePath + one batch of visibility rays) against the oracle's verdict pair by pair (= the reference's,
    test_ref_pin.py::test_same_topo_path_bit_exact)."""
    of = small_scene["field"]
    rng = np.random.default_rng(41)
    a, b = np.array([-7.5, -6.0]), np.array([7.0, 6.5])
    paths = []
    for _ in range(14):
        k = int(rng.integers(0, 4))
        mid = [a + (b - a) * t + rng.normal(size=2) * rng.choice([0.05, 1.0, 3.0]) for t in np.sort(rng.uniform(0.1, 0.9, k))]
        xy = np.clip(np.array([a] + mid + [b]), -9.5, 9.5)
        paths.append(np.concatenate([xy, np.zeros((len(xy), 1))], axis=1))
    pairs = np.array([(i, j) for i in range(len(paths)) for j in range(i + 1, len(paths))])
    for crit in (False, True):
        got = gpu_scene.sameTopoPaths(paths, pairs, 0.0, crit)
        exp = np.array([of.same_topo_path(paths[i], paths[j], 0.0, crit) for i, j in pairs])
        assert np.array_equal(got, exp)
    assert 0 < exp.sum() < len(exp)


def test_solvers_of_different_capacity_coexist(gpu_scene):
    """Kernel attributes (dynamic shared memory) are per kernel, not per solver: a small solver created after a
    large one must not break the large one, and results do not depend on what else was created."""
    import topay_b200 as tp
    from topay_b200 import scenes
    paths, bv, ba = scenes.short_candidates(2, 7)
    big = tp.MomaTrajOpt(gpu_scene, max_cand=2, max_pieces=64)
    a = big.optimizeTrajBatch(paths, bv, ba)
    small = tp.MomaTrajOpt(gpu_scene, max_cand=2, max_pieces=16)
    b = small.optimizeTrajBatch(paths, bv, ba)
    c = big.optimizeTrajBatch(paths, bv, ba)
    for r in (b, c):
        assert np.array_equal(a["evals"], r["evals"]) and np.array_equal(a["cost"], r["cost"])
        assert np.array_equal(a["T"][:, :16], r["T"][:, :16])


def test_spare_warp_does_not_reevaluate_the_end_node(gpu_scene):
    """K < K-hat: node 2K belongs to the piece's own segment. The warp that rounds k_penalty's grid up to whole
    blocks used to run as an end-node task and write gnode[K] a second time (a race with last-bit effects);
    its footprint was the end-node scratch, which must now stay untouched."""
    import ctypes as C
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()      # int_K = 12 -> K-hat = 16, two pieces per warp
    paths, bv, ba = scenes.short_candidates(4, 7)
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=4, max_pieces=16, opt_param=opt, robot=rp)
    prep = [tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 16) for p in paths]
    assert any(((q["piece_num"] + 1) // 2) % 2 == 1 for q in prep)    # an odd number of piece groups occurs
    solver.evaluate(2, [q["piece_num"] for q in prep], [q["head_pva"] for q in prep], [q["tail_pva"] for q in prep],
                    [q["start_xy"] for q in prep], [q["end_xy"] for q in prep], [q["init_inner_xy"] for q in prep],
                    [q["x0"] for q in prep], alm_lambda=np.zeros((4, 2)), alm_rho=np.full((4, 2), 1e4))
    buf = np.full(4 * 16 * 54, np.nan)
    n = solver._l.topay_solver_debug_download(solver.h, 7, buf.ctypes.data_as(C.POINTER(C.c_double)), len(buf))
    assert n == len(buf) and np.all(buf == 0.0)
