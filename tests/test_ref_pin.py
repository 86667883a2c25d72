"""Pins the oracle restatement to the REFERENCE'S OWN CODE, bit for bit.

oracle/_ref/libtopay_ref.so is the reference's lbfgs.hpp, banded_system.hpp, minco.hpp (MinJerkOpt<9>)
and moma_param.h (getColliPts / getColliGrads) compiled unmodified from the reference's source tree against the
Eigen / ROS stand-ins of oracle/ref_stubs (oracle/Makefile target _ref, tests/ref_lib.py). The
oracle functions of the same rows (SURVEY §8a a3, a4, a5, a8, a9, a10, a11, a13, a14) must return
IDENTICAL doubles on the same inputs: `np.array_equal`, no tolerance. The one stated limit: the stand-in
sums reductions (dot, norm, sum) sequentially, as the oracle does; real Eigen's packet order may differ
in the last ulp of a reduction.

The reference is not part of this repository. Where the compiled reference is present every comparison runs
against it live. Elsewhere each comparison checks the oracle's output against a digest of the reference's output
on the same inputs, stored in tests/golden/ref_pin.json: SHA-256 over shape and float64 values (-0.0 and NaN
made canonical, so that equal outputs give equal digests), first 16 hex digits. Run with TOPAY_REF_PIN_RECORD=1 to
rewrite the file from the outputs the tests compare. The stored digests were taken from the oracle, whose sources
are unchanged since commit a4d73c2; with those sources all 39 comparisons passed live against the compiled
reference, so the oracle's outputs here are the reference's.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import ref_lib as R
from topay_b200._structs import LbfgsParams

LIVE = R.available()
RECORD = os.environ.get("TOPAY_REF_PIN_RECORD") == "1"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin.json")


def _digest(value):
    h = hashlib.sha256()
    for a in (value if isinstance(value, tuple) else (value,)):
        a = np.asarray(a, dtype=np.float64)
        a = np.ascontiguousarray(np.where(np.isnan(a), np.nan, a + 0.0))
        h.update(np.asarray(a.shape, dtype=np.int64).tobytes())
        h.update(a.tobytes())
    return h.hexdigest()[:16]


class _Pin:
    """pin(orc, ref, what): the oracle's output `orc` must equal the reference's. `ref` computes the reference's
    output (a thunk, called only where the compiled reference is present); a tuple is compared element by element.
    Returns the reference's output (live) or the oracle's (checked against the stored digest)."""

    def __init__(self, name, stored):
        self.name, self.stored, self.seen = name, stored, []

    def _next(self):
        i = len(self.seen)
        assert self.stored is not None, f"no stored reference outputs for {self.name}"
        assert i < len(self.stored), f"{self.name}: more comparisons than stored reference outputs"
        return self.stored[i]

    def __call__(self, orc, ref, what=""):
        if LIVE:
            val = ref()
            if isinstance(orc, tuple):
                assert len(val) == len(orc), what
                for k, (a, b) in enumerate(zip(val, orc)):
                    assert np.array_equal(a, b), (what, k)
            else:
                assert np.array_equal(val, orc), what
        else:
            val = orc
            if not RECORD:
                assert _digest(orc) == self._next(), (what, "differs from the reference's stored output")
        self.seen.append(_digest(val))
        return val

    def value(self, v):
        """A value the reference's run depends on (process state): live as given, elsewhere as stored."""
        if not LIVE and not RECORD:
            v = self._next()
        self.seen.append(v)
        return v


@pytest.fixture(scope="module")
def _stored():
    stored = {}
    if os.path.exists(GOLDEN):
        with open(GOLDEN) as f:
            stored = json.load(f)
    recorded = {}
    yield stored, recorded
    if RECORD:
        stored.update(recorded)
        with open(GOLDEN, "w") as f:
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(stored.items())) + "\n}\n")


@pytest.fixture
def pin(request, _stored):
    stored, recorded = _stored
    p = _Pin(request.node.name, stored.get(request.node.name))
    failed = request.session.testsfailed
    yield p
    recorded[request.node.name] = p.seen
    if not LIVE and not RECORD and request.session.testsfailed == failed:
        assert len(p.seen) == len(p.stored), f"{request.node.name}: stored reference outputs left unchecked"


def _lp(**kw):
    d = dict(mem_size=8, g_epsilon=1e-8, past=3, delta=1e-10, max_iterations=0, max_linesearch=64, min_step=1e-20,
             max_step=1e20, f_dec_coeff=1e-4, s_curv_coeff=0.9, cautious_factor=1e-6, machine_prec=1e-16)
    d.update(kw)
    return LbfgsParams(**d)


@pytest.mark.skipif(not LIVE, reason="inspects the compiled reference (oracle/_ref), which is not present")
def test_reference_sources_are_the_reference():
    assert b"/root/reference" in R.lib().ref_sources()


@pytest.mark.parametrize("n,p,q,m", [(6, 6, 6, 9), (18, 6, 6, 9), (60, 6, 6, 9), (384, 6, 6, 9), (40, 2, 3, 1), (25, 4, 1, 5)])
def test_banded_system_bit_exact(oracle, pin, n, p, q, m):
    """a4: factorizeLU / solve / solveAdj (banded_system.hpp:66-145), incl. exact zeros inside the band."""
    rng = np.random.default_rng(n * 31 + p)
    A = np.zeros((n, n))
    for i in range(n):
        for j in range(max(0, i - p), min(n, i + q + 1)):
            A[i, j] = rng.normal() if rng.random() > 0.25 else 0.0   # the `!= 0.0` skips matter
        A[i, i] = 6.0 + rng.random()
    B = rng.normal(size=(n, m))
    for adj in (False, True):
        ref = pin(oracle.banded_solve(A, p, q, B, adj), lambda: R.banded_solve(A, p, q, B, adj), adj)
        assert np.abs((A.T if adj else A) @ ref - B).max() < 1e-9


@pytest.mark.parametrize("N", [1, 2, 3, 8, 17, 64])
def test_minjerk_generate_and_backprop_bit_exact(oracle, pin, N):
    """a3, a5, a11: MinJerkOpt<9>::generate, getTrajJerkCost, calJerkGradCT, calGradCTtoQT (minco.hpp:824-1069)."""
    rng = np.random.default_rng(100 + N)
    ew = np.array([0.33] + [1.0] * 8)
    head, tail = rng.normal(size=(9, 3)), rng.normal(size=(9, 3))
    inner, T = rng.normal(size=(max(N - 1, 0), 9)), rng.uniform(0.3, 2.5, N)
    pin(tuple(oracle.minco_generate(N, ew, head, tail, inner, T)),
        lambda: tuple(R.minco_generate(N, ew, head, tail, inner, T)), "coeff, jerk, gdC_jerk, gdT_jerk")
    gdC, gdT = rng.normal(size=(6 * N, 9)), rng.normal(size=N)
    pin(tuple(oracle.minco_backprop(N, ew, head, tail, inner, T, gdC, gdT)),
        lambda: tuple(R.minco_backprop(N, ew, head, tail, inner, T, gdC, gdT)), "gdP, gdTail, gdT")


def test_robot_constants_are_the_reference_constructor(oracle, pin):
    """a10 + the constants of moma_param.h:36-144 as its constructor evaluates them."""
    rp = oracle.robot_defaults()
    names = ("colli_length", "colli_points", "colli_radius", "joint_pos_max", "relative_t", "relative_R",
             "collision_matrix", "limits")
    pin((np.array(rp.colli_length), np.array(rp.colli_points), np.array(rp.colli_point_radius),
         np.array(rp.joint_pos_limit_max), np.array(rp.relative_t), np.array(rp.relative_R).reshape(3, 3),
         np.array(rp.collision_matrix).reshape(12, 12),
         [rp.max_v, rp.max_a, rp.max_w, rp.max_dw, rp.chassis_colli_radius, rp.chassis_height]),
        lambda: tuple(R.robot_constants()[k] for k in names), names)
    # the product's defaults are the same table
    import topay_b200 as tp
    pp = tp.robot_params_default()
    assert bytes(pp) == bytes(rp)


def test_fk_and_adjoint_bit_exact(oracle, pin):
    """a8, a9: getColliPts / getColliGrads (moma_param.h:203-337) on random whole-body states."""
    rng = np.random.default_rng(5)
    rp = oracle.robot_defaults()
    for _ in range(200):
        pos = np.concatenate([rng.uniform(-8, 8, 2), rng.uniform(-np.pi, np.pi, 1), rng.uniform(-3, 3, 7)])
        a = pin(oracle.colli_pts(rp, pos), lambda: R.colli_pts(pos), "colli_pts")
        assert a.shape == (12, 4)
        g = rng.normal(size=(12, 3)) * (rng.random((12, 1)) > 0.3)
        pin(oracle.colli_grads(rp, pos, g), lambda: R.colli_grads(pos, g), "colli_grads")


@pytest.mark.parametrize("case", ["rosenbrock", "ring_wrap", "stage1_like", "stage2_like", "max_iter", "ls_fail", "g_eps"])
def test_lbfgs_bit_exact(oracle, pin, case):
    """a13, a14: lbfgs_optimize + line_search_lewisoverton (lbfgs.hpp:276-722): same return code, iterate,
    cost and evaluation count on chained-Rosenbrock problems, incl. a history ring that wraps many times
    (mem_size 4), the reference's early-accept (:327-330, past > 0), max_iterations and line-search failure."""
    rng = np.random.default_rng(sum(map(ord, case)))
    n, b = 40, 1.0
    kw = {}
    if case == "ring_wrap":
        n, kw = 120, dict(mem_size=4, past=0, g_epsilon=1e-9)
    elif case == "stage1_like":
        kw = dict(mem_size=256, g_epsilon=0.0, past=2, delta=1e-2, min_step=0.0, max_iterations=8000)
    elif case == "stage2_like":
        n, b, kw = 200, 5.0, dict(mem_size=256, g_epsilon=0.0, past=3, delta=1e-4, min_step=1e-32, max_iterations=8000)
    elif case == "max_iter":
        kw = dict(max_iterations=7, past=0)
    elif case == "ls_fail":
        b, kw = 50.0, dict(max_linesearch=2, past=0)
    elif case == "g_eps":
        kw = dict(g_epsilon=1e-3, past=0)
    p = _lp(**kw)
    a, c, x0 = rng.uniform(0.5, 2.0, n), rng.normal(size=n), rng.normal(size=n)
    if case == "ls_fail":
        x0 = 3.0 * x0
    r_orc, x_orc, f_orc, it_orc, ev_orc = oracle.lbfgs_test_problem(a, c, b, p, x0)
    trace = []

    def ref():
        r_ref, x_ref, f_ref, it_ref, ev_ref, tr = R.lbfgs_test_problem(a, c, b, p, x0, trace_cap=10000)
        trace.extend(tr)
        return r_ref, ev_ref, x_ref, f_ref

    r_ref, _, _, _ = pin((r_orc, ev_orc, x_orc, f_orc), ref, "return code, evaluations, x, f")
    # accepted iterations: one row of the reference's progress trace each; the oracle counts them
    iters = len(trace) if LIVE else it_orc
    if case == "ring_wrap":
        assert iters > 6 * p.mem_size      # the ring really wrapped
    if case == "max_iter":
        assert r_ref == -997 or iters == 7   # LBFGSERR_MAXIMUMITERATION
    if case == "ls_fail":
        assert r_ref == -1009 and iters > 5   # LBFGSERR_MAXIMUMLINESEARCH after some accepted iterations


# ------------------------------------------------------------------------------------------------------------------
# The reference's whole optimizer and map (moma_traj_opt.cpp, grid_map.cpp) against the oracle
@pytest.fixture(scope="module")
def ref_scene(oracle, small_scene):
    if not LIVE:
        return None
    g = R.GridMap(small_scene["desc"])
    g.set_cloud(small_scene["points"])
    return g


def test_gridmap_buffers_bit_exact(oracle, pin, small_scene, ref_scene):
    """a20, a21, a22: cloudCallback rasterisation + updateESDF (grid_map.cpp:543-578, 89-521): occupancy and all four
    signed ESDF buffers (flat, inflated, critical, 3-D) of the default 200 x 200 x 16 scene."""
    of = small_scene["field"]
    for which in (0, 2, 3):
        pin(of.download_occupancy(which), lambda: ref_scene.download_occupancy(which), ("occupancy", which))
    for which in range(4):
        pin(of.download(which), lambda: ref_scene.download(which), ("esdf", which))


@pytest.mark.parametrize("size,res", [((3.1, 2.3, 0.9), 0.1), ((1.0, 1.0, 0.5), 0.25), ((6.0, 4.0, 1.2), 0.2)])
def test_gridmap_ragged_grids_bit_exact(oracle, pin, size, res):
    """a20/a21 on small ragged grids incl. the accumulate-critical quirk (grid_map.cpp:719-722) over two scenes."""
    from topay_b200._structs import grid_desc
    d = grid_desc(map_size=size, resolution=res)
    g, of = R.GridMap(d) if LIVE else None, oracle.Field(d)
    rng = np.random.default_rng(int(size[0] * 10))
    for scene in range(2):
        pts = (rng.uniform(-0.5, 0.5, (60, 3)) * np.array(size) + np.array([0, 0, size[2] / 2])).astype(np.float32)
        if LIVE:
            g.set_cloud(pts, clear=1)
        of.clear(False)
        of.rasterize(pts)
        of.rebuild()
        for which in range(4):
            pin(of.download(which), lambda: g.download(which), (scene, which))


def test_gridmap_queries_bit_exact(oracle, pin, small_scene, ref_scene):
    """a17, a18, a19: getDisWithGradI2d/3d, getDistance2d/3d, isWholeBodyCollision (grid_map.h:256-725), incl.
    positions outside the map and on its border."""
    of = small_scene["field"]
    rng = np.random.default_rng(0)
    q = np.concatenate([rng.uniform(-10.5, 10.5, (20000, 2)), rng.uniform(-0.2, 1.8, (20000, 1))], axis=1)
    q[:50, 0] = 10.0 - 1e-4 * np.arange(50) / 25
    pin(tuple(of.query3d(q)), lambda: tuple(ref_scene.query3d(q)), "query3d")
    for which in range(3):
        pin(tuple(of.query2d(q[:, :2], which)), lambda: tuple(ref_scene.query2d(q[:, :2], which)), ("query2d", which))
    pin(of.distance3d(q), lambda: ref_scene.distance3d(q), "distance3d")
    pin(of.distance2d(q[:, :2]), lambda: ref_scene.distance2d(q[:, :2]), "distance2d")
    rp = oracle.robot_defaults()
    st = np.concatenate([rng.uniform(-9, 9, (3000, 2)), rng.uniform(-np.pi, np.pi, (3000, 1)), rng.uniform(-2, 2, (3000, 7))], axis=1)
    pin(of.whole_body_collision(rp, st), lambda: ref_scene.whole_body_collision(st), "whole_body_collision")


def _front_cases(rng, n):
    """Polylines as the topological front end produces them: 2-6 waypoints inside the 20 m map."""
    out = []
    for i in range(n):
        k = int(rng.integers(2, 7))
        raw = rng.uniform(-8.5, 8.5, (k, 2))
        if i % 5 == 0:
            raw[1] = raw[0] + np.array([0.3, 0.0])          # a segment shorter than one step
        if i % 7 == 0 and k > 2:
            raw[2] = raw[1] + (raw[1] - raw[0])               # a straight continuation (zero turn: dropped rows)
        out.append((raw, rng.uniform(-np.pi, np.pi), rng.uniform(-np.pi, np.pi)))
    return out


def test_dense_path_bit_exact(oracle, pin, ref_scene):
    """N2: GraphSearch::getDensePath (graph_search.cpp:119-176) — segment subdivision, turn-in-place rows, angle
    unwrapping against the previous row, the 1e-3 s filter — row count and every (x, y, theta, dt) bit for bit."""
    rng = np.random.default_rng(5)
    for raw, y0, y1 in _front_cases(rng, 60):
        for step in (1.414, 0.5):
            pin(oracle.dense_path(raw, step, y0, y1, 1.0, 1.25),
                lambda: R.dense_path(ref_scene, raw, step, y0, y1, 1.0, 1.25), step)


def test_line_visib_bit_exact(oracle, pin, small_scene, ref_scene):
    """N2: TopologyPRM::lineVisib (topo_prm.cpp:278-315) over the planner's RayCaster (raycast.cpp:253-346): verdict and
    blocking point of 4000 segments across the cuboids scene, inflated and critical map, several clearances."""
    of = small_scene["field"]
    rng = np.random.default_rng(6)
    p1 = np.concatenate([rng.uniform(-9.5, 9.5, (4000, 2)), np.zeros((4000, 1))], axis=1)
    p2 = p1 + np.concatenate([rng.normal(size=(4000, 2)) * rng.choice([0.05, 0.5, 3.0], (4000, 1)), np.zeros((4000, 1))], axis=1)
    p2[:, :2] = np.clip(p2[:, :2], -9.9, 9.9)
    p2[::50] = p1[::50]                     # degenerate rays (setInput returns false)
    for crit in (False, True):
        for thresh in (0.0, 0.1, 0.3):
            def ref():
                va, pa = R.line_visib(ref_scene, p1, p2, thresh, crit)
                return va, pa[~va]
            vb, pb = of.line_visib(p1, p2, thresh, crit)
            va, _ = pin((vb, pb[~vb]), ref, ("verdict, blocking point", crit, thresh))
            assert 0.05 < va.mean() < 0.98


def _topo_paths(rng, n):
    """Pairs of polylines between common end points, as the PRM's path search returns them: some hug each other (same
    class), some pass on different sides of obstacles."""
    out = []
    for i in range(n):
        a, b = rng.uniform(-8.5, 8.5, 2), rng.uniform(-8.5, 8.5, 2)
        paths = []
        for _ in range(2):
            k = int(rng.integers(0, 4))
            mid = [a + (b - a) * t + rng.normal(size=2) * rng.choice([0.05, 0.8, 2.5]) for t in np.sort(rng.uniform(0.1, 0.9, k))]
            xy = np.clip(np.array([a] + mid + [b]), -9.5, 9.5)
            paths.append(np.concatenate([xy, np.zeros((len(xy), 1))], axis=1))
        out.append(paths)
    return out


def test_same_topo_path_bit_exact(oracle, pin, small_scene, ref_scene):
    """N2: TopologyPRM::pathLength, discretizePath and sameTopoPath (topo_prm.cpp:424-506): lengths and the equally
    spaced points bit for bit, the equivalence verdict on 300 path pairs (inflated and critical map)."""
    of = small_scene["field"]
    rng = np.random.default_rng(8)
    pairs = _topo_paths(rng, 300)
    verdicts = []
    for p1, p2 in pairs:
        pin(oracle.path_length(p1), lambda: R.path_length(ref_scene, p1), "path_length")
        pt = int(rng.integers(2, 120))
        pin(oracle.discretize_path(p1, pt), lambda: R.discretize_path(ref_scene, p1, pt), "discretize_path")
        for crit in (False, True):
            a = pin(of.same_topo_path(p1, p2, 0.0, crit), lambda: R.same_topo_path(ref_scene, p1, p2, 0.0, crit),
                    ("same_topo_path", crit))
            verdicts.append(a)
    assert 0.05 < np.mean(verdicts) < 0.95


@pytest.mark.parametrize("int_K,pieces", [(12, 0), (5, 0), (32, 64)])
def test_cost_callbacks_bit_exact(oracle, pin, small_scene, ref_scene, int_K, pieces):
    """a2, a6, a7, a12: first/secondStageCostCallback (moma_traj_opt.cpp:817-955) = generate + jerk + the penalty loops
    (:957-1829) + calGradCTtoQT + the C2 maps: cost, gradient and coefficients IDENTICAL; stage 2 also the 13 per-term
    costs and final_xy_error. (Stage 1 never resets the reference's debug terms, so they are not compared there.)"""
    from topay_b200 import scenes
    of = small_scene["field"]
    opt, rp = oracle.opt_defaults(), oracle.robot_defaults()
    opt.int_K = int_K
    if pieces:
        opt.min_piece_num, opt.sample_interval = pieces, 1e9
        paths, bv, ba = scenes.synthetic_batch(2, 1234)
    else:
        paths, bv, ba = scenes.short_candidates(4, 7)
    ro = R.MomaTrajOpt(ref_scene, opt) if LIVE else None
    rng = np.random.default_rng(3)
    for c, p in enumerate(paths):
        q = oracle.prepare_candidate(opt, rp, p, bv[c], ba[c], 64)
        N = q["piece_num"]
        for x in (q["x0"], q["x0"] + 0.05 * rng.normal(size=len(q["x0"]))):
            for stage in (1, 2):
                lam, rho = np.array([0.3, -0.2]), np.array([1e4, 3e4])
                args = (stage, N, q["head_pva"], q["tail_pva"], q["start_xy"], q["end_xy"], q["init_inner_xy"][:N], lam, rho, x)

                def ref():
                    f_r, g_r, t_r, c_r, e_r = ro.eval_one(*args)
                    return (f_r, g_r, c_r, t_r, e_r) if stage == 2 else (f_r, g_r, c_r)
                f_o, g_o, t_o, c_o, e_o = oracle.eval_one(opt, rp, of, *args)
                pin((f_o, g_o, c_o, t_o, e_o) if stage == 2 else (f_o, g_o, c_o), ref, (c, stage))


def test_optimize_traj_bit_exact(oracle, pin, small_scene, ref_scene):
    """a1, a13-a16 + N1: MomaTrajOpt::optimizeTraj (moma_traj_opt.cpp:142-498) end to end — pre-processing, stage 1,
    the ALM loop — then getTraj / checkFeasible / printConstraintsSituations: same status, and the final cost,
    durations and all 6N x 9 coefficients IDENTICAL to the oracle's; same gate verdicts. The reference's 1.0 s wall
    clock is frozen and ros::ok() carries the deterministic round cap (oracle/ref_driver_full.cpp)."""
    from topay_b200 import scenes
    of = small_scene["field"]
    opt, rp = oracle.opt_defaults(), oracle.robot_defaults()
    paths, bv, ba = scenes.short_candidates(4, 7)
    ro = R.MomaTrajOpt(ref_scene, opt) if LIVE else None
    for c, p in enumerate(paths):
        def ref():
            a = ro.solve_one(p, bv[c], ba[c], alm_max_rounds=opt.alm_max_rounds)
            chk, prt, _ = ro.gate()
            return a["status"], a["piece_num"], a["cost"], a["T"], a["coeff"], a["final_xy_err"], chk, prt
        b = oracle.solve_one(opt, rp, of, p, bv[c], ba[c], max_pieces=16)
        start = np.array([p[0][0], p[0][1], p[0][2]])
        g = oracle.check_feasible(of, rp, [(b["T"], b["coeff"], start)])
        pin((b["status"], b["piece_num"], b["cost"], b["T"], b["coeff"], b["final_xy_err"], bool(g["feasible"][0]),
             bool(g["feasible_print"][0])), ref, ("status, piece_num, cost, T, coeff, final_xy_err, checkFeasible, "
                                                  "printConstraintsSituations", c))


# ------------------------------------------------------------------------------------------------------------------
# The reference's ROG-Map ESDF layer (esdf_map.cpp, counter_map.cpp, sliding_map.cpp, raycaster.cpp)
@pytest.mark.parametrize("half,box", [((26, 26, 9), (4.0, 4.0, 1.5)), ((12, 12, 5), (9.0, 9.0, 9.0))])
def test_rog_esdf_layer_bit_exact(oracle, pin, half, box):
    """a23, a24, N3 (ESDF side): mapSliding, updateGridCounter, updateESDF3D with the ring-wrapped fillESDF, the six
    lookups and evaluateEDT over a sequence of slides that wraps every axis, clipped and full update boxes, cells
    seen free again — counters, the four persistent buffers (distance_buffer, tmp_buffer1_, critical, flat) and every
    query IDENTICAL to the reference's own classes. (Square rings: on non-square rings the reference's 2-D combine
    walks y over the x bounds, esdf_map.cpp:398-405, i.e. out of the row — the oracle clips it, a stated deviation.)"""
    from topay_b200._structs import rog_desc
    d = rog_desc(half_prob_map_size_i=half, prob_resolution=0.1, esdf_resolution=0.1, local_update_box=box,
                 map_sliding_en=True)
    ref, orc = R.RogESDFMap(d) if LIVE else None, oracle.RogField(d)
    maps = (ref, orc) if LIVE else (orc,)
    pin((orc.size, orc.half, orc.half_box, orc.resolution), lambda: (ref.size, ref.half, ref.half_box, ref.resolution),
        "geometry")
    rng = np.random.default_rng(half[0])
    ext = np.array(half) * 0.1 * 0.8
    for step, odom in enumerate([(0.0, 0.0, 0.0), (0.43, -0.31, 0.12), (0.9, -0.7, 0.2), (-0.3, 0.4, -0.1), (2.5, 1.9, 0.5)]):
        for m in maps:
            m.slide(odom)
        pin(orc.origin_i, lambda: ref.origin_i, ("origin", step))
        hits = rng.uniform(-1, 1, (300, 3)) * ext + np.array(odom)
        for m in maps:
            m.update_counters(hits, np.full(300, 1), np.full(300, 3))      # UNKNOWN -> OCCUPIED
            if step == 2:
                m.update_counters(hits[:100], np.full(100, 3), np.full(100, 4))   # OCCUPIED -> KNOWN_FREE
        pin(tuple(orc.download_counters()), lambda: tuple(ref.download_counters()), ("counters", step))
        for m in maps:
            m.update_esdf(odom)
        for which in range(4):
            pin(orc.download(which), lambda: ref.download(which), (step, which))
        q = rng.uniform(-1, 1, (2000, 3)) * ext + np.array(odom)
        for kind in range(6):
            pin(tuple(orc.query(kind, q)), lambda: tuple(ref.query(kind, q)), (step, kind))
        pin(orc.evaluate_edt(q), lambda: ref.evaluate_edt(q), ("evaluateEDT", step))
        # isLineFree2d (esdf_map.cpp:122-152) on short rays
        s2 = rng.uniform(-1, 1, (200, 2)) * ext[:2] * 0.8 + np.array(odom[:2])
        e2 = s2 + rng.uniform(-0.6, 0.6, (200, 2))
        pin(orc.is_line_free2d(s2, e2, 0.05), lambda: ref.is_line_free2d(s2, e2, 0.05), ("isLineFree2d", step))


# ------------------------------------------------------------------------------------------------------------------
# The reference's ProbMap (prob_map.cpp) driving its ESDFMap from point clouds — row N3
def _scan_cloud(rng, pos, n, spread, walls):
    """A synthetic lidar frame: points on a few planes around the robot + far / high / low outliers + intensities."""
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = np.minimum(np.abs(walls[0] / np.where(np.abs(d[:, 0]) > 1e-3, d[:, 0], 1e-3)),
                   np.abs(walls[1] / np.where(np.abs(d[:, 1]) > 1e-3, d[:, 1], 1e-3)))
    r = np.minimum(r, rng.uniform(0.2, spread, n))
    pts = pos + d * r[:, None]
    pts[::17] += rng.normal(size=(len(pts[::17]), 3)) * 5.0          # far, above the ceiling, below the ground
    inten = rng.uniform(0, 100, (n, 1))
    return np.concatenate([pts, inten], axis=1).astype(np.float32)


@pytest.mark.parametrize("cfg", [
    dict(half=(20, 20, 8), res=0.1, esdf_res=0.1, box=(3.0, 3.0, 1.2), upd=(3.5, 3.5, 1.4), filt=1, batch=1, inten=-1, ray=True),
    dict(half=(16, 18, 6), res=0.1, esdf_res=0.2, box=(2.5, 2.5, 1.0), upd=(99.0, 99.0, 99.0), filt=3, batch=2, inten=30, ray=True),
    dict(half=(14, 14, 6), res=0.1, esdf_res=0.1, box=(2.0, 2.0, 1.0), upd=(2.0, 2.0, 1.0), filt=2, batch=1, inten=-1, ray=False,
         inf_step=2),
])
def test_prob_map_bit_exact(oracle, pin, cfg):
    """N3: ProbMap::updateProbMap over a sequence of clouds and poses — the point filters (intensity, every k-th),
    clipping to ceiling / ground / range / update box, the 3-D ray walks, batched hit / miss log-odds updates, the type
    transitions forwarded to the ESDF counter map, map sliding with resetCell, poses outside the map and outside the
    ceiling, the first-frame sphere clearing — occupancy_buffer_ (float log-odds), the ESDF counters and the four ESDF
    buffers IDENTICAL to the reference's own ProbMap + ESDFMap after every frame."""
    from topay_b200._structs import prob_desc, rog_desc
    d = rog_desc(half_prob_map_size_i=cfg["half"], prob_resolution=cfg["res"], esdf_resolution=cfg["esdf_res"],
                 local_update_box=cfg["box"], map_sliding_en=True)
    p = prob_desc(ray_range=(0.3, 2.4), virtual_ceil_height=0.62, virtual_ground_height=-0.48,
                  local_update_box=cfg["upd"], map_sliding_thresh=0.25, point_filt_num=cfg["filt"],
                  batch_update_size=cfg["batch"], intensity_thresh=cfg["inten"], raycasting_en=cfg["ray"],
                  inflation_resolution=cfg["res"], inflation_step=cfg.get("inf_step", 1))
    ref = R.RogProbMap(d, p) if LIVE else None
    of = oracle.RogField(d)
    orc = oracle.RogProb(of, d, p)
    pin((orc.size, of.size), lambda: (ref.size, ref.esdf.size), "sizes")
    orc.set_first_frame(pin.value(R.RogProbMap.first_frame_pending()))
    rng = np.random.default_rng(cfg["half"][1])
    poses = [(0.0, 0.0, 0.0), (0.05, 0.02, 0.0), (0.31, -0.22, 0.05), (0.33, -0.2, 0.05), (0.9, 0.7, 0.1),
             (0.9, 0.7, 0.9), (9.0, 9.0, 0.0), (9.1, 9.0, 0.0), (8.7, 9.3, -0.1)]
    seen_occ = seen_free = False
    for step, pos in enumerate(poses):
        cloud = _scan_cloud(rng, np.array(pos), 700, 3.0, (1.3, 1.7))
        if LIVE:
            ref.update(cloud, pos)
        R.RogProbMap._first_done = True
        orc.update(cloud, pos)
        b, ob = orc.download()
        pin((b, ob), lambda: ref.download(), ("occupancy, origin", step))
        seen_occ, seen_free = seen_occ or bool((b > 0).any()), seen_free or bool((b < 0).any())
        pin(tuple(of.download_counters()), lambda: tuple(ref.esdf.download_counters()), ("counters", step))
        if cfg["half"][0] == cfg["half"][1]:        # square rings only (the 2-D combine quirk, see above)
            for which in range(4):
                pin(of.download(which), lambda: ref.esdf.download(which), (step, which))
    assert seen_occ and (seen_free or not cfg["ray"])
