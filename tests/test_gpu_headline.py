"""GPU parity at the HEADLINE configuration (BASELINE configs[2]: 64 pieces x int_K 32) and of the pieces of the
device solve the short reference-scale tests cannot reach: the full-history L-BFGS two-loop, the slot pool, and the
BASELINE-size field. The oracle is bit-identical to the reference's own code (tests/test_ref_pin.py)."""
import ctypes as C
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu_scene(small_scene):
    import topay_b200 as tp
    gm = tp.GridMap(small_scene["desc"], device=0)
    gm.regenerateMap(small_scene["points"])
    yield gm
    gm.close()


def _two_loop(S, Y, ys, g, end, bound, m, ys_new, yy_new):
    """lbfgs.hpp:691-710 verbatim: d = -g, first loop newest -> oldest, scale by ys/yy, second loop back."""
    d = -g.copy()
    alpha = np.zeros(m)
    j = end
    for _ in range(bound):
        j = (j + m - 1) % m
        alpha[j] = S[j].dot(d) / ys[j]
        d += (-alpha[j]) * Y[j]
    d *= ys_new / yy_new
    for _ in range(bound):
        beta = Y[j].dot(d) / ys[j]
        d += (alpha[j] - beta) * S[j]
        j = (j + 1) % m
    return d


@pytest.mark.parametrize("n", [52, 160, 161, 632])
@pytest.mark.parametrize("bound0,end0", [(0, 0), (0, 200), (6, 6), (6, 2), (254, 254), (255, 255), (256, 0), (256, 131),
                                         (256, 255)])
def test_lbfgs_direction_full_history(gpu_scene, n, bound0, end0):
    """a13: the device's paired, TMA-streamed two-loop (one launch of k_cand<L-BFGS> through
    topay_solver_debug_direction) against the reference recursion on the same (S, Y, g): histories of 1, 7, 255 and
    256 pairs, ring positions that wrap, the single-warp (n <= 160) and block-wide (n >= 161) variants, odd and even
    loop lengths. <= 1e-9 relative to |d|."""
    import topay_b200 as tp
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    m = opt.s2_lbfgs.mem_size
    assert m == 256
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=1, max_pieces=64, opt_param=opt, robot=rp)
    rng = np.random.default_rng(n * 1000 + bound0 * 3 + end0)
    S = rng.normal(size=(m, n)) * np.exp(rng.normal(size=(m, 1)))          # rows of very different scale
    A = np.exp(rng.normal(size=n))                                         # SPD diagonal "Hessian"
    Y = S * A + 0.05 * rng.normal(size=(m, n)) * np.abs(S).mean(axis=1, keepdims=True)
    ys = np.einsum("ij,ij->i", S, Y)
    assert (ys > 0).all()
    xp, gp = rng.normal(size=n), rng.normal(size=n)
    s_new = 0.3 * rng.normal(size=n)
    x, g = xp + s_new, gp + s_new * A + 0.01 * rng.normal(size=n)
    d = np.zeros(n)
    b_out, e_out = C.c_int32(), C.c_int32()
    dp = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))
    rc = solver._l.topay_solver_debug_direction(solver.h, n, bound0, end0, dp(S), dp(Y), dp(ys), dp(x), dp(xp), dp(g), dp(gp),
                                                dp(d), C.byref(b_out), C.byref(e_out))
    assert rc == 0
    # the reference's update (lbfgs.hpp:657-689): the new pair goes to row end0, then bound and end advance
    S2, Y2, ys2 = S.copy(), Y.copy(), ys.copy()
    S2[end0], Y2[end0] = x - xp, g - gp
    ys_new, yy_new = Y2[end0].dot(S2[end0]), Y2[end0].dot(Y2[end0])
    ys2[end0] = ys_new
    bound, end = min(bound0 + 1, m), (end0 + 1) % m
    assert (b_out.value, e_out.value) == (bound, end)
    exp = _two_loop(S2, Y2, ys2, g, end, bound, m, ys_new, yy_new)
    assert np.abs(d - exp).max() <= 1e-9 * np.abs(exp).max(), (np.abs(d - exp).max(), np.abs(exp).max())
    solver.close()


def test_pool_results_do_not_depend_on_the_slot_count(gpu_scene):
    """Continuous batching: 32 candidates through 32, 8 and 3 slots — the queue hands candidates to whichever slot
    frees first, yet every candidate's result is bit-identical (a candidate's arithmetic never depends on its slot or
    on its neighbours), all slots stay busy, and the per-plan winners of optimizeTrajPlans equal the flat solve's."""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths, bv, ba = scenes.short_candidates(32, 11)
    res = {}
    for ns in (32, 8, 3):
        s = tp.MomaTrajOpt(gpu_scene, max_cand=32, max_pieces=16, opt_param=opt, robot=rp, n_slots=ns)
        res[ns] = s.optimizeTrajBatch(paths, bv, ba)
        st = s.stats()
        assert res[ns]["evals"].sum() <= st["slot_ticks"] <= res[ns]["evals"].sum() + 32 * 16 * 2
        if ns == 3:
            assert res[ns]["evals"].sum() / st["slot_ticks"] > 0.97          # slots never idle while work waits
            plans = [(paths[i:i + 8], bv[i:i + 8], ba[i:i + 8]) for i in range(0, 32, 8)]
            rp_ = s.optimizeTrajPlans(plans)
            for i in range(4):
                sub = {k: res[32][k][8 * i:8 * i + 8] for k in ("status", "duration", "cost")}
                ok = np.flatnonzero(sub["status"] == 1)
                assert rp_["plan_best_by_duration"][i] == (ok[np.argmin(sub["duration"][ok])] if len(ok) else -1)
            assert np.array_equal(rp_["cost"], res[32]["cost"])
        s.close()
    for ns in (8, 3):
        for k in ("status", "lbfgs_code", "evals", "iters", "alm_rounds", "cost", "T", "coeff", "x", "final_xy_err"):
            assert np.array_equal(res[32][k], res[ns][k]), (ns, k)


def test_two_lanes_give_the_single_lane_results(gpu_scene, monkeypatch):
    """Large pools run their slots as two lanes (two parallel branches of the tick graph, each with its own live
    lists, one shared queue and store). Forced onto a small pool: 32 candidates through 9 and 2 slots split into
    lanes of 5 + 4 and 1 + 1 — every candidate's result bit-identical to the single-lane run, the gate and the
    device-side selection included."""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths, bv, ba = scenes.short_candidates(32, 11)
    plans = [(paths[i:i + 8], bv[i:i + 8], ba[i:i + 8]) for i in range(0, 32, 8)]
    res, win = {}, {}
    for lanes, ns in ((1, 9), (2, 9), (2, 2)):
        monkeypatch.setenv("TOPAY_LANE_MIN_SLOTS", "2" if lanes == 2 else "0")
        s = tp.MomaTrajOpt(gpu_scene, max_cand=32, max_pieces=16, opt_param=opt, robot=rp, n_slots=ns)
        res[lanes, ns] = s.optimizeTrajBatch(paths, bv, ba)
        st = s.stats()
        assert res[lanes, ns]["evals"].sum() <= st["slot_ticks"]
        assert st["eval_launches"] == lanes * st["ticks"]
        win[lanes, ns] = s.planWinners(plans, use_gate=True)
        s.close()
    for key in ((2, 9), (2, 2)):
        for k in ("status", "lbfgs_code", "evals", "iters", "alm_rounds", "cost", "T", "coeff", "x", "final_xy_err"):
            assert np.array_equal(res[1, 9][k], res[key][k]), (key, k)
        for a, b in zip(win[1, 9], win[key]):
            assert (a is None) == (b is None)
            if a is not None:
                assert a["index"] == b["index"]
                for k, v in a.items():
                    if isinstance(v, np.ndarray):
                        assert np.array_equal(v, b[k]), (key, k)


@pytest.mark.parametrize("lanes", [1, 2])
def test_tick_cap_marks_unfinished_candidates(gpu_scene, monkeypatch, lanes):
    """The hard cap on ticks (a runaway guard; forced here through TOPAY_MAX_TICKS): candidates still solving when it
    strikes — in a slot of either lane, or still waiting in the queue — come back with status 0 and the distinct
    code TOPAY_LBFGSERR_TICK_CAP; candidates that had finished keep their results."""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths, bv, ba = scenes.short_candidates(24, 11)
    monkeypatch.setenv("TOPAY_LANE_MIN_SLOTS", "2" if lanes == 2 else "0")
    s = tp.MomaTrajOpt(gpu_scene, max_cand=24, max_pieces=16, opt_param=opt, robot=rp, n_slots=6)
    full = s.optimizeTrajBatch(paths, bv, ba)
    monkeypatch.setenv("TOPAY_MAX_TICKS", "160")
    cut = s.optimizeTrajBatch(paths, bv, ba)
    monkeypatch.delenv("TOPAY_MAX_TICKS")
    s.close()
    capped = cut["lbfgs_code"] == tp.LBFGSERR_TICK_CAP
    assert capped.any() and (cut["status"][capped] == 0).all()
    assert capped[6:].sum() >= 12                  # most of the queue never reached a slot in 160 ticks
    done = ~capped
    for k in ("status", "lbfgs_code", "evals", "cost", "T"):
        assert np.array_equal(cut[k][done], full[k][done]), k
    assert (full["evals"][done] <= 160).all()


def test_scenarios_with_their_own_fields_share_one_solve():
    """BASELINE configs[4]: the candidates of several scenarios, each with its own field, in ONE upload
    (topay_solver_assign_fields). Every scenario's winner, trajectory and gate verdicts are bit-identical to solving that
    scenario alone against its field — also when the plans are handed over in another order. (16 slots run as one
    lane; test_gpu_launch_paths.py::test_sweep_pool_in_two_split_lanes runs a sweep in two lanes.)"""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    n_sc, n_c = 5, 6
    fields, plans, alone = [], [], []
    for sc in range(n_sc):
        g = tp.GridMap(tp.grid_desc())
        g.regenerateMap(scenes.tables_scene(70 + sc)[0] if sc % 2 == 0 else scenes.cuboids_scene(70 + sc)[0])
        fields.append(g)
        plans.append(scenes.short_candidates(n_c, 3000 + sc))
        one = tp.MomaTrajOpt(g, max_cand=n_c, max_pieces=16, opt_param=opt, robot=rp)
        alone.append((one.planWinners([plans[sc]], use_gate=True)[0], {k: v.copy() for k, v in one.constraints.items()}))
        one.close()
    pool = tp.MomaTrajOpt(fields[0], max_cand=n_sc * n_c, max_pieces=16, opt_param=opt, robot=rp, n_slots=16)
    for order in (list(range(n_sc)), [3, 0, 4, 2, 1]):
        got = pool.planWinners([plans[i] for i in order], use_gate=True, fields=[fields[i] for i in order])
        gate = pool.constraints
        for pos, sc in enumerate(order):
            w, (a, ag) = got[pos], alone[sc]
            assert (w is None) == (a is None)
            if w is not None:
                assert w["index"] == a["index"]
                for k, v in a.items():
                    if isinstance(v, np.ndarray):
                        assert np.array_equal(v, w[k]), (sc, k)
            for k in ("feasible", "feasible_print"):
                assert np.array_equal(gate[k][pos * n_c:(pos + 1) * n_c], ag[k]), (sc, k)
    # back to the solver's own field
    pool.assign_fields(None, None)
    back = pool.planWinners([plans[0]], use_gate=True)[0]
    assert (back is None) == (alone[0][0] is None) and (back is None or back["index"] == alone[0][0]["index"])
    pool.close()
    for g in fields:
        g.close()


def test_headline_config_solve_against_the_oracle(gpu_scene, small_scene, oracle):
    """The headline workload itself: the first 4 candidates of scenes.synthetic_batch(256, 1234) at 64 pieces x
    int_K 32, solved on the device and by the oracle (= the reference, bit for bit). The solve is chaotic — the
    oracle with its interior waypoints perturbed by 1e-15 relative already lands elsewhere — so the stated tolerance
    is: same success status; ALM rounds within 1; the first 15 accepted L-BFGS iterations replay the oracle's
    (same k, same line-search count, f within 1e-9); final cost, duration, base-path length inside the oracle's own
    perturbation band widened 3x (at least +-9 %); clearances within 0.15 m; BOTH gate verdicts (checkFeasible and
    printConstraintsSituations, planner.cpp:877-880) equal to the oracle's on its own trajectory."""
    import topay_b200 as tp
    from topay_b200 import scenes
    n = 4
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    paths, bv, ba = scenes.synthetic_batch(256, 1234)
    paths, bv, ba = paths[:n], bv[:n], ba[:n]
    of = small_scene["field"]
    solver = tp.MomaTrajOpt(gpu_scene, max_cand=n, max_pieces=64, opt_param=opt, robot=rp)
    solver.set_trace(20000)
    res = solver.optimizeTrajBatch(paths, bv, ba)
    gate, _ = solver.checkFeasibleBatch()
    gate = {k: v.copy() for k, v in gate.items()}
    exact, pert = [None] * n, [None] * n

    def work(c):
        exact[c] = oracle.solve_one(opt, rp, of, paths[c], bv[c], ba[c], max_pieces=64, trace=True)
        pp = paths[c].copy()
        pp[1:-1] *= (1 + 1e-15)
        pert[c] = oracle.solve_one(opt, rp, of, pp, bv[c], ba[c], max_pieces=64)

    th = [threading.Thread(target=work, args=(c,)) for c in range(n)]
    [t.start() for t in th]
    [t.join() for t in th]
    radii = np.array([rp.colli_point_radius[i] for i in range(16) if rp.colli_points[i] != 0.0])

    def metrics(T, coeff, start):
        g = oracle.check_feasible(of, rp, [(T, coeff, start)])
        seq = oracle.traj_car_seq([(T, coeff, start)])[0]
        length = np.linalg.norm(np.diff(seq[:, :2], axis=0), axis=1).sum()
        return g, length

    for c in range(n):
        o, p = exact[c], pert[c]
        assert res["status"][c] == o["status"] == 1 and res["piece_num"][c] == o["piece_num"] == 64
        assert abs(int(res["alm_rounds"][c]) - o["alm_rounds"]) <= 1
        tg, tc = solver.trace(c), o["trace"]
        m = 15
        assert np.array_equal(tg[:m, 2:], tc[:m, 2:])
        assert np.abs(tg[:m, 0] - tc[:m, 0]).max() <= 1e-9 * np.abs(tc[:m, 0]).max()
        start = paths[c][0, :3]
        go, len_o = metrics(o["T"], o["coeff"], start)
        gp_, len_p = metrics(p["T"], p["coeff"], start)
        N = 64
        gd, len_d = metrics(res["T"][c, :N], res["coeff"][c, :6 * N], start)
        for name, dev, a, b in (("cost", res["cost"][c], o["cost"], p["cost"]),
                                ("duration", res["duration"][c], o["duration"], p["duration"]),
                                ("length", len_d, len_o, len_p)):
            lo, hi = min(a, b), max(a, b)
            w = max(hi - lo, 0.03 * hi)
            assert lo - 3 * w <= dev <= hi + 3 * w, (c, name, dev, a, b)
        assert np.linalg.norm(res["final_xy_err"][c]) < opt.alm_tolerance
        # clearances of the device trajectory (device gate) against the oracle's on its trajectory
        assert abs(gate["min_dist"][c] - go["min_dist"][0]) <= 0.15
        arm_d = (gate["min_dist_mani"][c, :len(radii)] - radii).min()
        arm_o = (go["min_dist_mani"][0, :len(radii)] - radii).min()
        assert abs(arm_d - arm_o) <= 0.15
        # both verdicts of the success gate: device gate on the device trajectory == oracle gate on the same
        # trajectory (exact), and == the oracle's verdict on its own trajectory
        assert gate["feasible"][c] == gd["feasible"][0] and gate["feasible_print"][c] == gd["feasible_print"][0]
        assert gate["feasible"][c] == go["feasible"][0] and gate["feasible_print"][c] == go["feasible_print"][0]
    solver.close()


@pytest.mark.parametrize("dims", [(800, 800, 80), (803, 803, 83)])
def test_baseline_size_field_bit_exact(oracle, dims):
    """a20/a21 at BASELINE configs[3] size: the whole 800 x 800 x 80 grid (and the odd-sized 803 x 803 x 83 one)
    against the oracle — the integer squared-distance grids of both signs, all four signed ESDF buffers, bit for bit."""
    import topay_b200 as tp
    from topay_b200 import scenes
    size = tuple((d - 0.5) * 0.05 for d in dims)       # GridMap::init takes ceil(size / resolution)
    desc = tp.grid_desc(map_size=size, resolution=0.05)
    gm = tp.GridMap(desc)
    assert gm.voxel_num == dims
    pts, _ = scenes.cuboids_scene(7, size_x=40.0, size_y=40.0, scale=2.0)
    gm.regenerateMap(pts)
    of = oracle.Field(desc)
    of.rasterize(pts)
    of.rebuild()
    assert np.array_equal(gm.getOccBuffer3d(), of.download_occupancy(3))
    for which in (3, 0, 1, 2):
        assert np.array_equal(gm._download(which), of.download(which)), which
    sqp, sqn = gm.getSqDist(3)
    osp, osn = of.download_sqdist(3)
    assert np.array_equal(sqp, osp) and np.array_equal(sqn, osn)
    gm.close()


def test_device_side_selection_and_winner_download(gpu_scene, small_scene, oracle):
    """planner.cpp:999-1010 on the device (topay_solver_select): per-plan winners by duration and by cost equal the
    host rule applied to the full download (first success, replaced only by a strictly shorter duration), with and
    without the success gate; the single-candidate download equals the batch download's row; planWinners returns
    exactly those candidates while only the winners cross the bus."""
    import topay_b200 as tp
    from topay_b200 import scenes
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    plans = [scenes.short_candidates(8, 40 + i) for i in range(5)]
    plans[2] = (plans[2][0][:3], plans[2][1][:3], plans[2][2][:3])          # a ragged plan
    s = tp.MomaTrajOpt(gpu_scene, max_cand=40, max_pieces=16, opt_param=opt, robot=rp, n_slots=16)
    r = s.optimizeTrajPlans(plans)
    off = r["plan_offset"].astype(np.int32)
    gate, _ = s.checkFeasibleBatch()
    gate = {k: v.copy() for k, v in gate.items()}

    def host_pick(ok, val):
        best = -1
        for c in range(len(ok)):
            if ok[c] and (best < 0 or val[c] < val[best]):
                best = c
        return best

    for use_gate in (False, True):
        bd, bc = s.select(off, use_gate)
        for i in range(len(plans)):
            sl = slice(off[i], off[i + 1])
            ok = r["status"][sl] == 1
            if use_gate:
                ok = ok & (gate["feasible_print"][sl] != 0)
            assert bd[i] == host_pick(ok, r["duration"][sl]) and bc[i] == host_pick(ok, r["cost"][sl]), (use_gate, i)
        if not use_gate:
            assert np.array_equal(bd, r["plan_best_by_duration"]) and np.array_equal(bc, r["plan_best_by_cost"])
    one = s.download_candidate(int(off[1]) + 2)
    for k in ("status", "lbfgs_code", "piece_num", "iters", "evals", "alm_rounds", "cost", "duration", "T", "coeff",
              "final_xy_err", "x"):
        assert np.array_equal(one[k], r[k][off[1] + 2]), k
    # ties go to the lowest index: the same plan twice in one upload picks its first copy
    twice = [(plans[0][0] + plans[0][0], np.concatenate([plans[0][1]] * 2), np.concatenate([plans[0][2]] * 2))]
    r2 = s.optimizeTrajPlans(twice)
    bd2, bc2 = s.select()
    assert 0 <= bd2[0] < 8 and 0 <= bc2[0] < 8 and np.array_equal(r2["cost"][:8], r2["cost"][8:])
    # the whole worker flow with only the winners on the bus
    bd_gate, _ = None, None
    w = s.planWinners(plans, use_gate=True)
    r3 = s.optimizeTrajPlans(plans)
    g3, _ = s.checkFeasibleBatch()
    for i, wi in enumerate(w):
        sl = slice(off[i], off[i + 1])
        exp = host_pick((r3["status"][sl] == 1) & (g3["feasible_print"][sl] != 0), r3["duration"][sl])
        assert (wi is None) == (exp < 0)
        if wi is not None:
            assert wi["index"] == exp and np.array_equal(wi["coeff"], r3["coeff"][off[i] + exp])
    s.upload(*[np.concatenate(x) if not isinstance(x[0], list) else sum(x, []) for x in
               ([p[0] for p in plans], [p[1] for p in plans], [p[2] for p in plans])])
    assert s.d2h_bytes >= 0
    s.close()
