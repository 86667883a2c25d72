"""Streaming sessions on a ROG solver whose ring keeps changing (topay_solver_stream_set_snapshots), and the gate of a
trajectory on the ring (topay_traj_check_feasible_rog).

The ring is test_gpu_grid_geometry's slid 63 x 43 x 15 ring at 0.2 m over a 0.1 m probability map, its wrap running
through the candidates. While plans are live it slides, its counters change, it is rebuilt, and ProbMap frames update
it. With snapshots every plan must be bit-identical (results, gate metrics from stream_take, both winners) to the same
plan solved alone through the batch API by a ROG solver on the ring as it was at the plan's submit; that solve runs
right before the submit, on the same ring. Every loop that waits for plans is bounded."""
import numpy as np
import pytest

from test_gpu_stream import MAX_ADVANCES, RESULT_KEYS, _poll, _take
from test_gpu_stream_grace import ZEROED, _assert_same, _refused, _solo

pytestmark = pytest.mark.gpu

PLAN = 6
ODOM = np.array([5.0, 3.3, 0.4])


def _desc():
    import topay_b200 as tp
    return tp.rog_desc(half_prob_map_size_i=(60, 40, 12), prob_resolution=0.1, esdf_resolution=0.2,
                       map_sliding_en=True)


def _cells(dev, seed, lo, hi, odom):
    from topay_b200 import scenes
    pts, _ = scenes.cuboids_scene(seed, size_x=11.0, size_y=7.0, scale=0.5)
    pts = pts.astype(np.float64) + np.array([odom[0], odom[1], 0.0])
    pts = pts[np.all((pts > lo + 0.01) & (pts < hi - 0.01), axis=1)]
    return (np.unique(np.floor(pts / dev.resolution).astype(np.int64), axis=0) + 0.5) * dev.resolution


class _World:
    """The ring (and optionally the oracle's copy), built and slid as test_gpu_grid_geometry's, and the changes it goes
    through while plans solve: steps[k]() moves it to its next state."""

    def __init__(self, orc=None):
        import topay_b200 as tp
        from test_gpu_rog import OCC, UNK
        self.dev, self.orc = tp.ESDFMap(_desc()), orc
        self.dev.mapSliding(ODOM)
        res, half = self.dev.resolution, (np.array(self.dev.map_size_i) - 1) // 2
        self.wrap = (half[:2] + 1) * res                            # first world coordinate of ring cell 0
        self.lo = (np.array(self.dev.local_map_origin_i) - half) * res
        self.hi = (np.array(self.dev.local_map_origin_i) + half + 1) * res
        self.cells = _cells(self.dev, 5, self.lo, self.hi, ODOM)
        self._counters(self.cells, UNK, OCC)
        self._esdf(ODOM)
        self.odom = ODOM.copy()
        self.prob = None
        self.steps = [self._more_obstacles, self._slide, self._prob_frame, self._clear_some, self._prob_frame]

    def _counters(self, cells, a, b):
        self.dev.updateGridCounter(cells, a, b)
        if self.orc is not None:
            self.orc.update_counters(cells, np.full(len(cells), a), np.full(len(cells), b))

    def _esdf(self, odom):
        self.dev.updateESDF3D(odom)
        if self.orc is not None:
            self.orc.update_esdf(odom)

    def _more_obstacles(self):      # counter update + updateESDF3D
        from test_gpu_rog import OCC, UNK
        extra = _cells(self.dev, 11, self.lo, self.hi, ODOM)
        self._counters(extra, UNK, OCC)
        self._esdf(self.odom)

    def _slide(self):               # a slide (counters only), then a rebuild around the new position
        self.odom = self.odom + np.array([0.4, 0.2, 0.0])
        self.dev.mapSliding(self.odom)
        self._esdf(self.odom)

    def _clear_some(self):          # obstacles seen free again + updateESDF3D
        from test_gpu_rog import FREE, OCC
        self._counters(self.cells[::3], OCC, FREE)
        self._esdf(self.odom)

    def _prob_frame(self):          # ProbMap.updateProbMap: rays, counters and updateESDF3D in one call
        import topay_b200 as tp
        if self.prob is None:
            self.prob = tp.ProbMap(self.dev, tp.prob_desc(ray_range=(0.3, 6.0), inflation_resolution=0.1))
            self.seed = 20
        self.seed += 1
        from topay_b200 import scenes
        pts, _ = scenes.cuboids_scene(self.seed, size_x=9.0, size_y=6.0, scale=0.6)
        pts = pts.astype(np.float64)[:: 4] + np.array([self.odom[0] - 4.5, self.odom[1] - 3.0, 0.0])
        cloud = np.concatenate([pts, np.zeros((len(pts), 1))], axis=1).astype(np.float32)
        self.prob.updateProbMap(cloud, self.odom)

    def close(self):
        if self.prob is not None:
            self.prob.close()
        self.dev.close()


def _plans(world, n, seed):
    """n plans of PLAN 8-waypoint candidates, 2-4 m long, whose footprints straddle the wrap in x and in y."""
    from topay_b200 import scenes
    rng = np.random.default_rng(seed)
    plans = []
    for _ in range(n):
        paths = []
        while len(paths) < PLAN:
            a = world.wrap + rng.uniform([-1.8, -1.6], [-0.4, -0.4])
            b = world.wrap + rng.uniform([0.4, 0.4], [1.8, 1.6])
            if rng.random() < 0.5:
                a, b = b, a
            if 2.0 <= np.linalg.norm(b - a) <= 4.0:
                paths.append(scenes.scurve_candidate(rng, a, b, 8, 0.3))
        plans.append((paths, np.zeros((PLAN, 10, 2)), np.zeros((PLAN, 10, 2))))
    return plans


def _differs(a, b):
    return any(not np.array_equal(a["res"][k], b["res"][k]) for k in RESULT_KEYS) or \
        any(not np.array_equal(a["gate"][k], b["gate"][k]) for k in a["gate"])


def _advance_and_take(s, n, got, ids, wins):
    for _ in range(n):
        s.stream_advance(1)
        for pid in _poll(s, wins):
            _take(s, pid, got, ids, wins)


def _drain(s, got, ids, wins):
    for _ in range(MAX_ADVANCES):
        live = s.stream_advance(1)
        for pid in _poll(s, wins):
            _take(s, pid, got, ids, wins)
        if live == 0 and not ids:
            return
    raise AssertionError(f"plans still unfinished after {MAX_ADVANCES} advances: {sorted(ids)}")


# A ROG solver has a slot per store row (pools are dense-only), so slot scarcity is not a case here; two lanes and timed
# mode are.
CONFIGS = {
    "status": dict(G=None, gate=False),
    "gate": dict(G=None, gate=True),
    "grace zero": dict(G=0, gate=False),
    "grace middle, gate": dict(G=40, gate=True),
    "two lanes": dict(G=None, gate=True, n_slots=512, max_cand=512),
    "timed": dict(G=None, gate=True, n_slots=16, timed=True),
}


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_plans_keep_the_ring_of_their_submit(cfg):
    """Two plans per ring state, the session advancing one or two batches between states, so that plans are live while
    the ring slides, its counters change, it is rebuilt and ProbMap frames update it: every plan bit-identical to its
    solo solve on the ring of its submit. At least one plan solves differently on the final ring, so a session that
    read the live ring would fail."""
    import topay_b200 as tp
    c = CONFIGS[cfg]
    world = _World()
    n = 2 * (len(world.steps) + 1)
    plans = _plans(world, n, 31)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    s = tp.MomaTrajOpt(world.dev, max_cand=c.get("max_cand", n * PLAN), max_pieces=16, n_slots=c.get("n_slots"))
    if c.get("timed"):
        s.set_timed(True)
    s.stream_begin(use_gate=c["gate"], grace_evals=c["G"], snapshots=len(world.steps) + 1)
    exp, got, ids, wins = [None] * n, [None] * n, {}, {}
    i = 0
    for step in range(len(world.steps) + 1):
        for _ in range(2):
            exp[i] = _solo(one, plans[i], c["G"], int(c["gate"]))
            ids[s.stream_submit(*plans[i])] = i
            i += 1
        _advance_and_take(s, 1 + step % 2, got, ids, wins)
        if step < len(world.steps):
            world.steps[step]()
    _drain(s, got, ids, wins)
    st = s.stats()
    s.stream_end()
    final = [_solo(one, p, c["G"], int(c["gate"])) for p in plans]
    one.close()
    s.close()
    world.close()
    for p in range(n):
        _assert_same(got[p], exp[p], c["gate"], (cfg, p))
    changed = [p for p in range(n) if _differs(exp[p], final[p])]
    assert changed, "no plan solves differently on the final ring: the ring changes test nothing"
    if c.get("n_slots") == 512:
        assert st["eval_launches"] == 2 * st["ticks"], st
    if c["G"] is not None:
        print(f"{cfg}: {sum(int((e['res']['lbfgs_code'] == tp.LBFGSERR_PLAN_GRACE).sum()) for e in exp)} cancelled")
    print(f"{cfg}: {len(changed)} of {n} plans differ on the final ring")


def test_snapshots_are_shared_and_held_until_take():
    """One snapshot: two submits on an unchanged ring share it; after an update a third submit is refused with
    TOO_LARGE and changes nothing (no plan id, no store rows); once both plans are taken, three plans on the new ring
    fill the whole store with the three plan ids, and everything matches its solo solve."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_TOO_LARGE
    world = _World()
    plans = _plans(world, 3, 47)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    s = tp.MomaTrajOpt(world.dev, max_cand=3 * PLAN, max_pieces=16)
    s.stream_begin(use_gate=True, snapshots=1)
    exp = [_solo(one, p, None, 1) for p in plans[:2]]
    got, ids, wins = [None] * 5, {}, {}
    ids[s.stream_submit(*plans[0])] = 0
    ids[s.stream_submit(*plans[1])] = 1                   # the same ring: no second snapshot needed
    world.steps[0]()
    _refused(ERR_TOO_LARGE, s.stream_submit, *plans[2])
    _refused(ERR_TOO_LARGE, s.stream_submit, *plans[2])   # still held: taken plans only release it
    _drain(s, got, ids, wins)
    exp += [_solo(one, p, None, 1) for p in (plans[2], plans[0], plans[1])]
    pids = set()
    for k, p in enumerate((plans[2], plans[0], plans[1])):
        pid = s.stream_submit(*p)                          # all 3 x PLAN rows: the refusals took none
        pids.add(pid)
        ids[pid] = 2 + k
    assert pids == {0, 1, 2}, pids
    _drain(s, got, ids, wins)
    s.stream_end()
    one.close()
    s.close()
    world.close()
    for p in range(5):
        _assert_same(got[p], exp[p], True, ("shared", p))


def test_a_stop_in_a_snapshot_session():
    """Plans on three ring states, one stopped mid-run: each of its candidates is either bit-identical to its solo
    result or cancelled, the ones that finished a batch before the stop are kept, and the other plans are
    bit-identical to their solo solves on the ring of their submit."""
    import topay_b200 as tp
    world = _World()
    plans = _plans(world, 6, 53)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    s = tp.MomaTrajOpt(world.dev, max_cand=len(plans) * PLAN, max_pieces=16)
    s.stream_begin(use_gate=True, snapshots=3)
    exp, got, ids, wins, pid = [None] * 6, [None] * 6, {}, {}, []
    for k in range(3):
        for i in (2 * k, 2 * k + 1):
            exp[i] = _solo(one, plans[i], None, 1)
            pid.append(s.stream_submit(*plans[i]))
            ids[pid[-1]] = i
        if k < 2:
            world.steps[k]()
    mid = max(range(6), key=lambda p: int(exp[p]["res"]["evals"].max()) - int(exp[p]["res"]["evals"].min()))
    b = max(2, -(-int(exp[mid]["res"]["evals"].min()) // 16) + 1)
    assert 16 * b + 32 < int(exp[mid]["res"]["evals"].max()), (b, exp[mid]["res"]["evals"])
    for k in range(1, MAX_ADVANCES):
        live = s.stream_advance(1)
        reported = _poll(s, wins)
        if k == b:
            assert pid[mid] not in wins, "the plan finished before its stop"
            s.stream_stop(pid[mid])
        for q in reported:
            _take(s, q, got, ids, wins)
        if live == 0 and not ids:
            break
    assert not ids
    s.stream_end()
    one.close()
    s.close()
    world.close()
    g, u = got[mid], exp[mid]
    kept = g["res"]["lbfgs_code"] != tp.LBFGSERR_PLAN_GRACE
    for c in range(PLAN):
        if kept[c]:
            for k in RESULT_KEYS:
                assert np.array_equal(g["res"][k][c], u["res"][k][c]), ("stopped plan", c, k)
            for k, v in u["gate"].items():
                assert np.array_equal(g["gate"][k][c], v[c]), ("stopped plan", c, "gate", k)
        else:
            assert g["res"]["status"][c] == 0 and g["res"]["piece_num"][c] == u["res"]["piece_num"][c]
            assert all(not np.any(g["res"][k][c]) for k in ZEROED) and all(not np.any(v[c]) for v in g["gate"].values())
    finished = u["res"]["evals"] <= 16 * (b - 1)
    assert finished.any() and (~kept).any()
    assert kept[finished].all(), "a candidate that finished before the stop was cancelled"
    for p in range(6):
        if p != mid:
            _assert_same(got[p], exp[p], True, ("other plans", p))


def test_snapshots_off_again():
    """After stream_set_snapshots(0) with every plan taken, a plan reads the live ring, matches its solo solve, and
    its advances and take cost as many launches as in a session that never had snapshots."""
    import topay_b200 as tp
    world = _World()
    plans = _plans(world, 2, 59)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    launches = {}
    for mode in ("off again", "never on"):
        s = tp.MomaTrajOpt(world.dev, max_cand=2 * PLAN, max_pieces=16)
        s.stream_begin(use_gate=True, snapshots=2 if mode == "off again" else 0)
        got, ids, wins = [None] * 2, {}, {}
        if mode == "off again":
            ids[s.stream_submit(*plans[0])] = 0
            _drain(s, got, ids, wins)
            s.stream_set_snapshots(0)
        exp = _solo(one, plans[1], None, 1)
        before = s.stats()["kernel_launches"]
        ids[s.stream_submit(*plans[1])] = 1
        _drain(s, got, ids, wins)
        launches[mode] = s.stats()["kernel_launches"] - before
        s.stream_end()
        s.close()
        _assert_same(got[1], exp, True, mode)
    one.close()
    world.close()
    assert launches["off again"] == launches["never on"], launches


def test_refusals(small_scene):
    """stream_set_snapshots on a dense solver or with n < 0: INVALID_ARG; outside a session or while a plan is
    untaken: NOT_READY. A submit, and the ring gate, on a ring never updated: NOT_READY."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_INVALID_ARG, ERR_NOT_READY
    world = _World()
    plans = _plans(world, 1, 61)
    s = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    _refused(ERR_NOT_READY, s.stream_set_snapshots, 1)
    s.stream_begin(use_gate=False)
    _refused(ERR_INVALID_ARG, s.stream_set_snapshots, -1)
    s.stream_set_snapshots(1)
    pid = s.stream_submit(*plans[0])
    _refused(ERR_NOT_READY, s.stream_set_snapshots, 0)
    got, ids, wins = [None], {pid: 0}, {}
    for _ in range(MAX_ADVANCES):
        s.stream_advance(1)
        if _poll(s, wins):
            break
    _refused(ERR_NOT_READY, s.stream_set_snapshots, 2)   # finished but not taken: it still holds its snapshot
    _take(s, pid, got, ids, wins)
    s.stream_set_snapshots(2)
    s.stream_end()
    _refused(ERR_NOT_READY, s.stream_set_snapshots, 1)
    s.close()
    gm = tp.GridMap(small_scene["desc"], device=0)
    gm.regenerateMap(small_scene["points"])
    d = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16)
    d.stream_begin()
    _refused(ERR_INVALID_ARG, d.stream_set_snapshots, 1)
    d.stream_end()
    d.close()
    gm.close()
    fresh = tp.ESDFMap(_desc())
    r = tp.MomaTrajOpt(fresh, max_cand=PLAN, max_pieces=16)
    r.stream_begin(snapshots=1)
    _refused(ERR_NOT_READY, r.stream_submit, *plans[0])
    r.stream_end()
    traj = tp.MomaTraj(np.ones(2), np.zeros((12, 9)), np.array([6.0, 4.0, 0.0]))
    _refused(ERR_NOT_READY, r.checkFeasible, traj)
    r.close()
    fresh.close()
    world.close()


def test_gate_on_the_ring(oracle):
    """topay_traj_check_feasible_rog on a ROG solver's trajectories equals its solver-resident gate bit for bit, and the
    oracle's gate on the same ring within test_gpu_traj's tolerances, for trajectories across the wrap and the same
    ones moved so that they leave the local map; checkFeasible / printConstraintsSituations work on a ROG solver."""
    import topay_b200 as tp
    from test_gpu_grid_geometry import _assert_same as _close_to
    from test_gpu_rog import _compare
    orc = oracle.RogField(_desc())
    orc.slide(ODOM)
    world = _World(orc)
    _compare(world.dev, orc, "ring for the gate")
    plans = _plans(world, 1, 67)
    rp = tp.robot_params_default()
    s = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16, robot=rp)
    s.optimizeTrajBatch(*plans[0])
    batch, _ = s.checkFeasibleBatch()
    batch = {k: v.copy() for k, v in batch.items()}
    trajs = [s.getTraj(c) for c in range(PLAN)]
    verdict = s.checkFeasible(trajs)
    for k, v in batch.items():
        assert np.array_equal(s.constraints[k], v), k
    assert np.array_equal(verdict, batch["feasible"].astype(bool))
    assert np.array_equal(s.printConstraintsSituations(trajs), batch["feasible_print"].astype(bool))
    assert s.checkFeasible(trajs[0]) == bool(batch["feasible"][0])
    away = world.hi[:2] - world.wrap + np.array([0.3, 0.2])       # the wrap crossing moved past the map's edge
    moved = [tp.MomaTraj(t.durations, t.coeff, t.start_se2 + np.array([away[0], away[1], 0.0])) for t in trajs]
    both = trajs + moved
    s.checkFeasible(both)
    oracle.use_rog(orc)
    try:
        exp = oracle.check_feasible(None, rp, [t._tuple() for t in both])
    finally:
        oracle.use_rog(None)
    _close_to(s.constraints, exp)
    s.close()
    world.close()


def test_snapshots_turned_on_mid_session():
    """A plain ROG session solves plans on the live ring (its batch graphs are captured), then snapshots go on and the
    same plans (no larger piece count, so the same launch grids) are submitted again; the ring goes through every
    change while they are live. Each plan of both waves is bit-identical to its solo solve on the ring of its submit,
    and some plan solves differently on the final ring, so replaying graphs captured on the live ring would fail."""
    import topay_b200 as tp
    world = _World()
    plans = _plans(world, 4, 71)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    s = tp.MomaTrajOpt(world.dev, max_cand=len(plans) * PLAN, max_pieces=16)
    s.stream_begin(use_gate=True)
    got, exp = [], []
    for wave in range(2):
        if wave == 1:
            s.stream_set_snapshots(2)
        g, ids, wins = [None] * len(plans), {}, {}
        exp.append([_solo(one, p, None, 1) for p in plans])
        for i, p in enumerate(plans):
            ids[s.stream_submit(*p)] = i
        _advance_and_take(s, 1, g, ids, wins)
        if wave == 1:
            assert ids, "every plan finished in one batch: the ring changes test nothing"
            for step in world.steps:
                step()
        _drain(s, g, ids, wins)
        got.append(g)
    s.stream_end()
    final = [_solo(one, p, None, 1) for p in plans]
    one.close()
    s.close()
    world.close()
    for wave in range(2):
        for p in range(len(plans)):
            _assert_same(got[wave][p], exp[wave][p], True, ("wave", wave, p))
    assert any(_differs(exp[1][p], final[p]) for p in range(len(plans))), "no plan differs on the final ring"


def test_a_polled_plan_holds_its_snapshot_until_take():
    """One snapshot: a plan that has been polled but not taken still holds it, so after a ring update a submit is
    refused with TOO_LARGE, and the take's gate, which reads the snapshot again, matches the solo solve on the ring of
    the plan's submit. After the take a submit on the new ring goes through and matches its own solo solve."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_TOO_LARGE
    world = _World()
    plans = _plans(world, 2, 73)
    one = tp.MomaTrajOpt(world.dev, max_cand=PLAN, max_pieces=16)
    s = tp.MomaTrajOpt(world.dev, max_cand=2 * PLAN, max_pieces=16)
    s.stream_begin(use_gate=True, snapshots=1)
    exp = [_solo(one, plans[0], None, 1)]
    got, ids, wins = [None, None], {s.stream_submit(*plans[0]): 0}, {}
    for _ in range(MAX_ADVANCES):
        s.stream_advance(1)
        if _poll(s, wins):
            break
    assert list(wins) == list(ids), "the plan was not reported"
    for step in world.steps:
        step()
    _refused(ERR_TOO_LARGE, s.stream_submit, *plans[1])
    _take(s, next(iter(ids)), got, ids, wins)
    exp.append(_solo(one, plans[1], None, 1))
    ids[s.stream_submit(*plans[1])] = 1
    _drain(s, got, ids, wins)
    s.stream_end()
    one.close()
    s.close()
    world.close()
    for p in range(2):
        _assert_same(got[p], exp[p], True, ("held until take", p))
