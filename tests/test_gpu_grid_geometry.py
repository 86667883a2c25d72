"""Field geometry: every consumer of a dense field on grids other than the default 200 x 200 x 16 one, against the
oracle. On a square grid nx == ny, so a transposed stride, an x bound used for y, a wrong clamp of the last cell or
a MULTI kernel that reads the solver's own geometry instead of its candidate's all go unseen.

Grids (cell counts given, map_size = (dims - 0.3) * res: ceil(map_size / res) is unambiguous and the last cell
sticks out past max_boundary, so the upper-edge clamp is reached inside the map):

  A  134 x  80 x 13 @ 0.1   wider than deep
  B  192 x 289 x 40 @ 0.05  deeper than wide, chassis_colli_radius 0.3, chassis_height 0.25
  C  155 x  90 x 12 @ 0.2   coarse
  D    7 x 300 x  5 @ 0.1   degenerate strip (random occupancy, queries only)

Covered: the query kernels, the predicates and coarse lookups, the visibility rays and the whole-body check on A-D
(and topay_field_query3d_dev on B); one evaluation of both stages on A-C with candidates along and across the
edges; solve, trace and gate on A; scenarios of four geometries in one MULTI solve; the benchmark's
800 x 800 x 80 field; the ROG-mode solver on a slid, non-square ring whose wrap runs through the candidates.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from test_gpu_parity import RESULT_KEYS, _check_eval_against_oracle, _eval_batch
from test_gpu_traj import _assert_same

pytestmark = pytest.mark.gpu

# id -> (dims, resolution, extra grid_desc arguments)
GRIDS = {
    "A": ((134, 80, 13), 0.1, {}),
    "B": ((192, 289, 40), 0.05, dict(chassis_colli_radius=0.3, chassis_height=0.25)),
    "C": ((155, 90, 12), 0.2, {}),
    "D": ((7, 300, 5), 0.1, {}),
}


def grid_spec(name):
    """(desc, lo, hi) of grid `name`: lo / hi are min_boundary / max_boundary as the library computes them."""
    from topay_b200._structs import grid_desc
    dims, res, kw = GRIDS[name]
    desc = grid_desc(map_size=tuple((d - 0.3) * res for d in dims), resolution=res, **kw)
    ms = np.array(desc.map_size[:])
    return desc, np.array([-ms[0] / 2.0, -ms[1] / 2.0, 0.0]), np.array([ms[0] / 2.0, ms[1] / 2.0, ms[2]])


def random_occupancy(dims, seed):
    """(occ3, occ2, occ2_critical) at 2 % fill: the strip D is too narrow for the cuboid generator's boxes."""
    rng = np.random.default_rng(seed)
    return ((rng.random(dims) < 0.02).astype(np.int8), (rng.random(dims[:2]) < 0.02).astype(np.int8),
            (rng.random(dims[:2]) < 0.02).astype(np.int8))


@pytest.fixture(scope="module")
def grids(oracle):
    """name -> dict(gm, of, desc, lo, hi, res, dims): the device field and the oracle field on the same input,
    checked bit-identical here so that the tests below compare lookups on equal buffers."""
    import topay_b200 as tp
    from topay_b200 import scenes
    out = {}
    for k, name in enumerate(GRIDS):
        dims, res, _ = GRIDS[name]
        desc, lo, hi = grid_spec(name)
        gm, of = tp.GridMap(desc), oracle.Field(desc)
        assert gm.voxel_num == of.dims == dims
        if name == "D":
            occ3, occ2, occ2c = random_occupancy(dims, 17)
            gm.loadMap(occ2, occ3, occ2c)
            of.set_occupancy(occ3, occ2, occ2c)
        else:
            ms = desc.map_size
            pts, _ = scenes.cuboids_scene(90 + k, size_x=ms[0], size_y=ms[1], scale=np.sqrt(ms[0] * ms[1] / 400.0))
            gm.regenerateMap(pts)
            of.clear(False)
            of.rasterize(pts)
        of.rebuild()
        assert np.array_equal(gm.getOccBuffer3d(), of.download_occupancy(3)), name
        for which in (3, 0, 1, 2):
            assert np.array_equal(gm._download(which), of.download(which)), (name, which)
        out[name] = dict(gm=gm, of=of, desc=desc, lo=lo, hi=hi, res=res, dims=dims)
    yield out
    for g in out.values():
        g["gm"].close()


def _positions(g, rng, n):
    """Uniform over the map +-3 cells; a band of +-2 cells round each of the six faces; and points whose coordinates
    are cell centres, cell faces or the in-map cut-off (boundary -+ 1e-4) and its neighbouring doubles."""
    lo, hi, res, dims = g["lo"], g["hi"], g["res"], g["dims"]
    uniform = rng.uniform(lo - 3 * res, hi + 3 * res, (n, 3))
    band = rng.uniform(lo, hi, (n, 3))
    ax, side = rng.integers(0, 3, n), rng.integers(0, 2, n)
    band[np.arange(n), ax] = np.where(side == 0, lo[ax], hi[ax]) + rng.uniform(-2 * res, 2 * res, n)
    special = rng.uniform(lo, hi, (n, 3))
    for a in range(3):
        i = np.arange(-1, dims[a] + 2)
        cut = [v for b in (lo[a] + 1e-4, hi[a] - 1e-4) for v in (np.nextafter(b, -np.inf), b, np.nextafter(b, np.inf))]
        values = np.concatenate([lo[a] + (i + 0.5) * res, lo[a] + i * res, np.repeat(cut, 20)])
        pick = rng.random(n) < 0.7
        special[pick, a] = rng.choice(values, int(pick.sum()))
    return np.concatenate([uniform, band, special])


@pytest.mark.parametrize("name", list(GRIDS))
def test_field_api_against_the_oracle(grids, oracle, name):
    """Queries (values <= 1e-12, gradients <= 1e-11: FMA contraction only), predicates, Bresenham line checks, coarse
    lookups, visibility rays and the whole-body check on grid `name`, at points in, round and outside the map."""
    g = grids[name]
    gm, of, lo, hi, res, dims = g["gm"], g["of"], g["lo"], g["hi"], g["res"], g["dims"]
    rng = np.random.default_rng(sum(dims))
    pos = _positions(g, rng, 20000)
    p2 = pos[:, :2]
    inside = np.all((pos > lo + 1e-4) & (pos < hi - 1e-4), axis=1)
    assert 0.2 < inside.mean() < 0.9
    d0, g0 = of.query3d(pos)
    d1, g1 = gm.getDisWithGradI3d(pos)
    assert np.abs(d0 - d1).max() <= 1e-12 and np.abs(g0 - g1).max() <= 1e-11
    assert np.all(d1[~np.all((pos >= lo + 1e-4) & (pos <= hi - 1e-4), axis=1)] == 0.0)
    v0, v1 = of.distance3d(pos), gm.getDistance3d(pos)
    assert np.array_equal(v0 == 1e10, v1 == 1e10) and np.abs(v0 - v1).max() <= 1e-12
    for w, kw in ((0, {}), (1, dict(inflate=True)), (2, dict(critical=True))):
        d0, g0 = of.query2d(p2, w)
        d1, g1 = gm.getDisWithGradI2d(p2, **kw)
        assert np.abs(d0 - d1).max() <= 1e-12 and np.abs(g0 - g1).max() <= 1e-11, w
    v0, v1 = of.distance2d(p2), gm.getDistance2d(p2)
    assert np.array_equal(v0 == 1e10, v1 == 1e10) and np.abs(v0 - v1).max() <= 1e-12

    for thr in (0.0, 0.25, 0.4):
        for q, got in ((p2, gm.isCollision2d(p2, thr)), (pos, gm.isCollision3d(pos, thr))):
            exp = of.is_collision(q, thr)
            d = of.distance2d(q) if q.shape[1] == 2 else of.distance3d(q)
            near = np.abs(d - thr) < 1e-12
            assert np.array_equal(got[~near], exp[~near]) and 0 < exp.sum() < len(exp), (thr, q.shape[1])

    # segments: random ones, and ones from inside the map out through each of the four sides
    n = 4000
    a = rng.uniform(lo[:2] + res, hi[:2] - res, (n, 2))
    b = rng.uniform(lo[:2] - 3 * res, hi[:2] + 3 * res, (n, 2))
    side = np.arange(n) % 5
    for s in range(4):
        ax, sel = s % 2, side == s
        b[sel, ax] = (lo[ax] if s < 2 else hi[ax]) + (-1 if s < 2 else 1) * rng.uniform(0.01, 1.0, sel.sum())
    b[:40] = a[:40]
    for thr in (0.0, 0.3):
        got, exp = gm.isLineCollisionGrid2d(a, b, thr), of.line_collision2d(a, b, thr)
        assert np.array_equal(got, exp) and 0 < exp.sum() < len(exp), thr

    idx = rng.integers(-5, max(dims) + 6, (n, 2))
    for crit in (False, True):
        assert np.array_equal(gm.getDistCoarse2d(p2, crit), of.dist_coarse2d(p2, crit)), crit
        assert np.array_equal(gm.getDistCoarse2i(idx, crit), of.dist_coarse2i(idx, crit)), crit

    q1 = np.concatenate([pos[:n, :2], np.zeros((n, 1))], axis=1)
    q2 = q1 + np.concatenate([rng.normal(size=(n, 2)) * rng.choice([0.05, 0.5, 4.0], (n, 1)), np.zeros((n, 1))], axis=1)
    q2[::40] = q1[::40]
    for crit in (False, True):
        for thresh in (0.0, 0.25):
            vg, pg = gm.lineVisib(q1, q2, thresh, crit)
            vo, po = of.line_visib(q1, q2, thresh, crit)
            assert np.array_equal(vg, vo) and np.array_equal(pg[~vg], po[~vo]), (crit, thresh)

    # whole-body states with the base within 1 m of an edge, inside and outside
    from topay_b200 import scenes
    m = 4000
    xy = rng.uniform(lo[:2], hi[:2], (m, 2))
    side = rng.integers(0, 4, m)
    ax = side % 2
    xy[np.arange(m), ax] = np.where(side < 2, lo[ax], hi[ax]) + rng.uniform(-1.0, 1.0, m)
    states = np.concatenate([xy, rng.uniform(-3, 3, (m, 1)), np.stack([scenes.random_joints(rng) * 1.02 for _ in range(m)])],
                            axis=1)
    exp = of.whole_body_collision(oracle.robot_defaults(), states).astype(bool)
    got = gm.isWholeBodyCollision(states)
    assert (exp != got).mean() < 1e-3          # only threshold-grazing states may differ
    if name != "D":                            # the 0.67 m strip is narrower than the chassis: every state collides
        assert 0.05 < exp.mean() < 0.999


def test_query3d_on_device_pointers(grids):
    """topay_field_query3d_dev (the benchmark's resident-query path) on torch tensors: bit-identical to
    topay_field_query3d on grid B."""
    import torch
    from topay_b200 import _lib
    g = grids["B"]
    gm = g["gm"]
    pos = _positions(g, np.random.default_rng(5), 20000)
    d_host, g_host = gm.getDisWithGradI3d(pos)
    dev = f"cuda:{gm.device}"
    p = torch.from_numpy(pos).to(dev)
    dist = torch.full((len(pos),), np.nan, dtype=torch.float64, device=dev)
    grad = torch.full((len(pos), 3), np.nan, dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)              # the call is ordered on the field's stream only
    l = _lib.lib()
    _lib.check(l.topay_field_query3d_dev(gm.h, C.c_void_p(p.data_ptr()), len(pos), C.c_void_p(dist.data_ptr()),
                                         C.c_void_p(grad.data_ptr())), "query3d_dev")
    _lib.check(l.topay_field_sync(gm.h), "sync")
    assert np.array_equal(dist.cpu().numpy(), d_host) and np.array_equal(grad.cpu().numpy(), g_host)


def _edge_candidates(g, rng):
    """Guide paths inside the grid that run within 0.5 m of an edge or corner, that leave it through a side or a
    corner (sphere lookups out of the map read 0; those just inside hit the upper-edge clamp), and one inside."""
    from topay_b200 import scenes
    lo, hi = g["lo"][:2], g["hi"][:2]
    c = 0.5 * (lo + hi)
    ends = [((lo[0] + 0.4, lo[1] + 0.4), (lo[0] + 4.0, lo[1] + 0.45)),      # from the corner (min, min) along y = min
            ((hi[0] - 0.4, hi[1] - 0.4), (hi[0] - 0.45, hi[1] - 6.0)),      # from the corner (max, max) along x = max
            ((hi[0] - 2.0, c[1]), (hi[0] + 1.5, c[1] + 0.5)),              # out through x = max
            ((c[0], lo[1] + 2.0), (c[0] - 0.7, lo[1] - 1.5)),              # out through y = min
            ((lo[0] + 1.5, hi[1] - 1.5), (lo[0] - 1.0, hi[1] + 1.0)),      # out through the corner (min, max)
            ((c[0] - 1.0, c[1] - 0.3), (c[0] + 1.0, c[1] + 0.3))]          # inside
    return [scenes.scurve_candidate(rng, np.array(a), np.array(b), 8, lateral=0.3) for a, b in ends]


@pytest.mark.parametrize("K", [12, 32])
@pytest.mark.parametrize("name", ["A", "B", "C"])
def test_eval_at_the_edges(grids, oracle, name, K):
    """One evaluation of both stages against the oracle (tolerances of test_eval_parity) for a ragged batch of edge
    candidates on grid `name`; K-hat = 16 has no end-node warps, K-hat = 32 has them."""
    import topay_b200 as tp
    g = grids[name]
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K = K
    paths = _edge_candidates(g, np.random.default_rng(K + ord(name)))
    prep = [tp.prepare_candidate(opt, rp, p, np.zeros((10, 2)), np.zeros((10, 2)), 16) for p in paths]
    assert all(q["rc"] == 0 for q in prep) and len({q["piece_num"] for q in prep}) > 1
    solver = tp.MomaTrajOpt(g["gm"], max_cand=len(prep), max_pieces=16, opt_param=opt, robot=rp)
    worst = _check_eval_against_oracle(solver, g["of"], oracle, opt, rp, prep, K)
    # the edge candidates reach the chassis and sphere lookups
    ev = _eval_batch(solver, 2, prep, [q["x0"] for q in prep], np.zeros((len(prep), 2)), np.full((len(prep), 2), 1e4))
    assert (ev["terms"][:, 2] != 0).any() and (ev["terms"][:, 6] != 0).any()
    solver.close()
    print(f"grid {name}, K={K}: worst relative deviation from the oracle {worst:.2e}")


def _in_map_candidates(g, rng, n, margin=1.6, dist=(3.0, 6.0)):
    from topay_b200 import scenes
    lo, hi = g["lo"][:2] + margin, g["hi"][:2] - margin
    paths = []
    while len(paths) < n:
        a, b = rng.uniform(lo, hi), rng.uniform(lo, hi)
        if dist[0] <= np.linalg.norm(a - b) <= dist[1]:
            paths.append(scenes.scurve_candidate(rng, a, b, 8, 0.6))
    return paths, np.zeros((n, 10, 2)), np.zeros((n, 10, 2))


def test_solve_trace_and_gate_on_a_wide_grid(grids, oracle):
    """Grid A: a solve of 6 candidates replays the oracle's first accepted iterations (same k and line-search count,
    f within 1e-9) with the same status; the solver-resident gate on the device's trajectories, and the host-call
    gate on them plus a time-compressed copy moved so that its base reaches the last half-cell before max_boundary,
    equal the oracle's gate on the same trajectories (verdicts and sample counts exact, metrics <= 1e-10)."""
    import topay_b200 as tp
    from topay_b200.optimizer import MomaTraj
    g = grids["A"]
    of = g["of"]
    n = 6
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths, bv, ba = _in_map_candidates(g, np.random.default_rng(61), n)
    solver = tp.MomaTrajOpt(g["gm"], max_cand=n, max_pieces=16, opt_param=opt, robot=rp)
    solver.set_trace(4000)
    res = solver.optimizeTrajBatch(paths, bv, ba)
    exact = [None] * n

    def work(c):
        exact[c] = oracle.solve_one(opt, rp, of, paths[c], bv[c], ba[c], max_pieces=16, trace=True)

    th = [threading.Thread(target=work, args=(c,)) for c in range(n)]
    [t.start() for t in th]
    [t.join() for t in th]
    for c in range(n):
        o = exact[c]
        assert res["status"][c] == o["status"] and res["piece_num"][c] == o["piece_num"], c
        tg, tc = solver.trace(c), o["trace"]
        m = 8
        assert len(tg) >= m and len(tc) >= m, c
        assert np.array_equal(tg[:m, 2:], tc[:m, 2:]), c
        assert np.abs(tg[:m, 0] - tc[:m, 0]).max() <= 1e-9 * np.abs(tc[:m, 0]).max(), c
    assert res["status"].sum() >= 1
    trajs = [solver.getTraj(c) for c in range(n)]
    arrs, _ = solver.checkFeasibleBatch()
    _assert_same(arrs, oracle.check_feasible(of, rp, [t._tuple() for t in trajs]))
    # time-compressed by 3 (limits violated), moved along x until its base reaches max_boundary - 0.01 m
    base = trajs[int(np.flatnonzero(res["status"] == 1)[0])]
    N = len(base.durations)
    coeff = (base.coeff.reshape(N, 6, 9) * (3.0 ** np.arange(6))[None, :, None]).reshape(6 * N, 9)
    fast = MomaTraj(base.durations / 3.0, coeff, base.start_se2)
    shift = g["hi"][0] - 0.01 - fast.car_seq[:, 0].max()
    edge = MomaTraj(fast.durations, fast.coeff, fast.start_se2 + np.array([shift, 0.0, 0.0]))
    assert abs(edge.car_seq[:, 0].max() - (g["hi"][0] - 0.01)) < 1e-9
    cases = trajs + [edge]
    solver.checkFeasible(cases)
    exp = oracle.check_feasible(of, rp, [t._tuple() for t in cases])
    _assert_same(solver.constraints, exp)
    assert exp["feasible"][-1] == 0
    solver.close()


def test_scenarios_of_four_geometries_share_one_solve(grids, small_scene):
    """One scenario on each of A, B, C and the default grid, solved in one upload (k_penalty<MULTI> and k_feasible
    read each candidate's own geometry), plans handed over in two orders: every candidate's results, each plan's
    winner and both gate verdicts bit-identical to solving that scenario alone on its own field."""
    import topay_b200 as tp
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    default = tp.GridMap(small_scene["desc"])
    default.regenerateMap(small_scene["points"])
    lo, hi = np.array([-10.0, -10.0, 0.0]), np.array([10.0, 10.0, 1.6])
    geo = [grids["A"], grids["B"], grids["C"], dict(gm=default, lo=lo, hi=hi)]
    fields = [s["gm"] for s in geo]
    n_c = 6
    plans, alone = [], []
    for sc, s in enumerate(geo):
        plans.append(_in_map_candidates(s, np.random.default_rng(700 + sc), n_c))
        one = tp.MomaTrajOpt(s["gm"], max_cand=n_c, max_pieces=16, opt_param=opt, robot=rp)
        w = one.planWinners([plans[sc]], use_gate=True)[0]
        alone.append((w, {k: v.copy() for k, v in one.constraints.items()}, one.download()))
        one.close()
    assert sum(a[0] is not None for a in alone) >= 3
    pool = tp.MomaTrajOpt(fields[0], max_cand=len(geo) * n_c, max_pieces=16, opt_param=opt, robot=rp, n_slots=16)
    for order in ([0, 1, 2, 3], [2, 0, 3, 1]):
        got = pool.planWinners([plans[i] for i in order], use_gate=True, fields=[fields[i] for i in order])
        gate = {k: v.copy() for k, v in pool.constraints.items()}
        full = pool.download()
        # the second order puts other candidates into the store rows the first order used: what a row held before
        # must not show past the new candidate's pieces
        for c, N in enumerate(full["piece_num"]):
            assert not full["T"][c, N:].any() and not full["coeff"][c, 6 * N:].any(), c
        for pos, sc in enumerate(order):
            w, (a, ag, af) = got[pos], alone[sc]
            sl = slice(pos * n_c, (pos + 1) * n_c)
            for k in RESULT_KEYS:
                assert np.array_equal(full[k][sl], af[k]), (sc, k)
            assert (w is None) == (a is None), sc
            if w is not None:
                assert w["index"] == a["index"]
                for k, v in a.items():
                    if isinstance(v, np.ndarray):
                        assert np.array_equal(v, w[k]), (sc, k)
            for k in ("feasible", "feasible_print"):
                assert np.array_equal(gate[k][sl], ag[k]), (sc, k)
    pool.close()
    default.close()


def test_eval_on_the_benchmark_field(oracle):
    """The 800 x 800 x 80 field at 0.05 m built as bench.py's field probe builds it (integer grids not kept), its
    ESDF buffers bit-identical to the oracle's, and one evaluation per stage of the first 3 headline candidates
    (64 pieces x int_K 32) against the oracle on that field."""
    import topay_b200 as tp
    from topay_b200 import scenes
    desc = tp.grid_desc(map_size=(40.0, 40.0, 4.0), resolution=0.05)
    gm = tp.GridMap(desc)
    pts, _ = scenes.cuboids_scene(7, size_x=40.0, size_y=40.0, scale=2.0)
    gm.regenerateMap(pts)
    gm.set_keep_sqdist(False)
    gm.updateESDF()
    of = oracle.Field(desc)
    of.rasterize(pts)
    of.rebuild()
    for which in (3, 0, 1, 2):
        assert np.array_equal(gm._download(which), of.download(which)), which
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    paths, bv, ba = scenes.synthetic_batch(256, 1234)
    prep = [tp.prepare_candidate(opt, rp, paths[c], bv[c], ba[c], 64) for c in range(3)]
    assert all(q["piece_num"] == 64 for q in prep)
    solver = tp.MomaTrajOpt(gm, max_cand=3, max_pieces=64, opt_param=opt, robot=rp)
    worst = _check_eval_against_oracle(solver, of, oracle, opt, rp, prep, 1234)
    solver.close()
    gm.close()
    print(f"800x800x80 field: worst relative deviation from the oracle {worst:.2e}")


def test_solver_on_a_slid_non_square_rog_ring(oracle):
    """ROG mode on a 63 x 43 x 15 ring at 0.2 m (counters and ESDF coarser than the 0.1 m probability map) slid so
    that the ring's wrap (global cell 31 -> 32 in x, 21 -> 22 in y) runs through the candidates: buffers bit-exact
    after the update, one evaluation per stage within the test_eval_parity tolerances, and the solver-resident gate
    equal to the oracle's on the device's trajectories."""
    import topay_b200 as tp
    from topay_b200 import scenes
    from topay_b200.rog import ESDFMap
    from test_gpu_rog import OCC, UNK, _compare
    desc = tp.rog_desc(half_prob_map_size_i=(60, 40, 12), prob_resolution=0.1, esdf_resolution=0.2,
                       map_sliding_en=True)
    dev, orc = ESDFMap(desc), oracle.RogField(desc)
    res = dev.resolution
    assert dev.map_size_i == orc.size == (63, 43, 15) and res == 0.2
    odom = np.array([5.0, 3.3, 0.4])
    dev.mapSliding(odom)
    orc.slide(odom)
    assert dev.local_map_origin_i == orc.origin_i == (25, 16, 2)
    wrap = (np.array(orc.half[:2]) + 1) * res                 # first world coordinate of ring cell 0: (6.4, 4.4)
    lo = (np.array(orc.origin_i) - orc.half) * res            # the local map
    hi = (np.array(orc.origin_i) + orc.half + 1) * res
    assert np.all(lo[:2] < wrap - 2) and np.all(wrap + 2 < hi[:2])
    pts, _ = scenes.cuboids_scene(5, size_x=11.0, size_y=7.0, scale=0.5)
    pts = pts.astype(np.float64) + np.array([odom[0], odom[1], 0.0])
    pts = pts[np.all((pts > lo + 0.01) & (pts < hi - 0.01), axis=1)]
    cells = np.unique(np.floor(pts / res).astype(np.int64), axis=0)     # one counter increment per occupied cell
    centres = (cells + 0.5) * res
    dev.updateGridCounter(centres, UNK, OCC)
    orc.update_counters(centres, np.full(len(centres), UNK), np.full(len(centres), OCC))
    dev.updateESDF3D(odom)
    orc.update_esdf(odom)
    _compare(dev, orc, "slid ring")
    # 2-4 m candidates whose footprint straddles the wrap in x and in y
    rng = np.random.default_rng(9)
    paths = []
    while len(paths) < 6:
        a = wrap + rng.uniform([-1.8, -1.6], [-0.4, -0.4])
        b = wrap + rng.uniform([0.4, 0.4], [1.8, 1.6])
        if rng.random() < 0.5:
            a, b = b, a
        if 2.0 <= np.linalg.norm(b - a) <= 4.0:
            paths.append(scenes.scurve_candidate(rng, a, b, 8, 0.3))
    n = len(paths)
    bv, ba = np.zeros((n, 10, 2)), np.zeros((n, 10, 2))
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    solver = tp.MomaTrajOpt(dev, max_cand=n, max_pieces=16, opt_param=opt, robot=rp)
    assert solver.use_rog
    oracle.use_rog(orc)
    try:
        prep = [tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 16) for p in paths]
        worst = _check_eval_against_oracle(solver, None, oracle, opt, rp, prep, 9)
        res_ = solver.optimizeTrajBatch(paths, bv, ba)
        assert res_["status"].sum() >= 1
        arrs, _ = solver.checkFeasibleBatch()
        trajs = [solver.getTraj(c)._tuple() for c in range(n)]
        _assert_same(arrs, oracle.check_feasible(None, rp, trajs))
    finally:
        oracle.use_rog(None)
    solver.close()
    dev.close()
    print(f"slid ROG ring: worst relative deviation from the oracle {worst:.2e}")
