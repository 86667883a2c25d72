"""Streaming sessions (topay_solver_stream_*): plans submitted while the solve runs, each plan's winners handed back as
soon as that plan is done.

Every expectation is the same plan solved alone through the batch API on a fresh upload (upload, run, download,
check_feasible, select): per candidate every result field and every gate metric, per plan the winners by duration and
by cost, all bit for bit. Sessions are driven under several arrival schedules, slot counts, two lanes, timed mode,
recycled store rows, per-plan fields and a slid ROG ring. Every loop that waits for plans is bounded, so a defect
fails the test instead of hanging it."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RESULT_KEYS = ("status", "lbfgs_code", "piece_num", "iters", "evals", "alm_rounds", "cost", "duration", "T", "coeff",
               "final_xy_err", "x")
PLAN = 8
MAX_ADVANCES = 4000     # 64000 ticks: far more than any plan here needs


def _plans(n, seed0=7100, size=PLAN):
    """Reference-scale plans of `size` candidates (bench.latency_probe's kind: int_K 12, 3-10 pieces)."""
    from topay_b200 import scenes
    return [scenes.short_candidates(size, seed0 + p) for p in range(n)]


def _solo(solver, plan):
    """The plan solved alone through the batch API: results, gate metrics, winners with and without the gate."""
    solver.upload(*plan)
    solver.run()
    res = {k: v.copy() for k, v in solver.download().items() if k in RESULT_KEYS}
    gate, _ = solver.checkFeasibleBatch()
    win = {g: tuple(int(v[0]) for v in solver.select(None, use_gate=g)) for g in (False, True)}
    return dict(res=res, gate={k: v.copy() for k, v in gate.items()}, win=win)


def _solos(field, plans, max_cand=PLAN):
    import topay_b200 as tp
    s = tp.MomaTrajOpt(field, max_cand=max_cand, max_pieces=16)
    out = [_solo(s, p) for p in plans]
    s.close()
    return out


def _take(s, pid, got, ids, wins):
    """Takes plan `pid` (results with gate metrics) into got[plan index]."""
    r = s.stream_take(pid, gate=True)
    i = ids.pop(pid)
    got[i] = dict(res={k: r[k] for k in RESULT_KEYS}, gate=r["gate"], win=wins.pop(pid))


def _poll(s, wins):
    for pid, bd, bc in s.stream_poll():
        assert pid not in wins, ("plan reported twice", pid)
        wins[pid] = (bd, bc)
    return list(wins)


def _drain(s, got, ids, wins, take=True):
    """Advances until every submitted plan has been reported (and taken, with take)."""
    for _ in range(MAX_ADVANCES):
        live = s.stream_advance(1)
        done = _poll(s, wins)
        if take:
            for pid in done:
                _take(s, pid, got, ids, wins)
        if live == 0 and len(wins) == len(ids) and (not take or not ids):
            return
    raise AssertionError(f"plans still unfinished after {MAX_ADVANCES} advances: {sorted(ids)}")


def _stream(s, plans, schedule, use_gate, fields=None):
    """One session over `plans` under an arrival schedule; returns one dict per plan (results, gate, winners)."""
    got, ids, wins = [None] * len(plans), {}, {}
    s.stream_begin(use_gate=use_gate)

    def submit(i):
        pid = s.stream_submit(*plans[i], field=None if fields is None else fields[i])
        assert pid not in ids
        ids[pid] = i

    if schedule == "upfront":              # everything queued before the first batch
        for i in range(len(plans)):
            submit(i)
        _drain(s, got, ids, wins)
    elif schedule == "one_per_advance":    # one plan per batch, results taken as they come
        for i in range(len(plans)):
            submit(i)
            s.stream_advance(1)
            for pid in _poll(s, wins):
                _take(s, pid, got, ids, wins)
        _drain(s, got, ids, wins)
    elif schedule == "interleaved":        # bursts, polls between them, takes deferred by one round
        deferred, i, rng = [], 0, np.random.default_rng(3)
        for _ in range(MAX_ADVANCES):
            if i < len(plans):
                for _ in range(int(rng.integers(1, 4))):
                    if i < len(plans):
                        submit(i)
                        i += 1
            s.stream_advance(int(rng.integers(1, 3)))
            for pid in deferred:
                _take(s, pid, got, ids, wins)
            deferred = [p for p in _poll(s, wins) if p not in deferred]
            if i == len(plans) and not ids:
                break
            if i == len(plans) and len(wins) == len(ids):
                for pid in list(wins):
                    _take(s, pid, got, ids, wins)
                deferred = []
        assert not ids, "plans still unfinished"
    else:
        raise ValueError(schedule)
    s.stream_end()
    return got


def _assert_same(got, solo, use_gate, what):
    for p, (g, e) in enumerate(zip(got, solo)):
        for k in RESULT_KEYS:
            assert np.array_equal(g["res"][k], e["res"][k]), (what, p, k)
        for k, v in e["gate"].items():
            assert np.array_equal(g["gate"][k], v), (what, p, "gate", k)
        assert g["win"] == e["win"][use_gate], (what, p, "winners", g["win"], e["win"][use_gate])


@pytest.fixture(scope="module")
def gm(small_scene):
    import topay_b200 as tp
    g = tp.GridMap(small_scene["desc"], device=0)
    g.regenerateMap(small_scene["points"])
    yield g
    g.close()


@pytest.fixture(scope="module")
def ref(gm):
    """12 reference-scale plans of 8 and their solo batch solves."""
    plans = _plans(12)
    solo = _solos(gm, plans)
    assert sum(s["win"][True][0] >= 0 for s in solo) >= 6      # most plans have a gated winner
    return plans, solo


@pytest.mark.parametrize("schedule", ["upfront", "one_per_advance", "interleaved"])
def test_arrival_schedules(gm, ref, schedule):
    """Plans all queued before the first batch, one per batch, or in bursts with polls and deferred takes (8 slots,
    gate on): every plan bit-identical to its solo solve."""
    import topay_b200 as tp
    plans, solo = ref
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=8)
    _assert_same(_stream(s, plans, schedule, True), solo, True, schedule)
    st = s.stats()
    assert st["ticks"] > 0 and st["evals_total"] == sum(int(e["res"]["evals"].sum()) for e in solo)
    s.close()


@pytest.mark.parametrize("n_slots", [3, 8, None])
def test_slot_counts(gm, ref, n_slots):
    """3, 8 and all slots (gate off, plans in bursts): every plan bit-identical to its solo solve."""
    import topay_b200 as tp
    plans, solo = ref
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=n_slots)
    _assert_same(_stream(s, plans, "interleaved", False), solo, False, f"{n_slots} slots")
    s.close()


def test_two_lanes_refilled_after_a_drain(gm):
    """A 512-slot pool (two lanes, 256 slots each) starts empty; 33 plans (264 candidates, more than one lane holds)
    are refilled into both lanes, the pool drains completely, and the same 33 plans arrive again: both lanes are
    refilled a second time. Every plan of both waves is bit-identical to its solo solve."""
    import topay_b200 as tp
    plans = _plans(33, seed0=7300)
    solo = _solos(gm, plans)
    s = tp.MomaTrajOpt(gm, max_cand=2 * len(plans) * PLAN, max_pieces=16, n_slots=512)
    s.stream_begin(use_gate=True)
    for wave in range(2):
        got, ids, wins = [None] * len(plans), {}, {}
        for i, p in enumerate(plans):
            ids[s.stream_submit(*p)] = i
        _drain(s, got, ids, wins, take=False)           # every plan finished before any is taken
        assert s.stream_advance(1) == 0                 # fully drained
        for pid in list(wins):
            _take(s, pid, got, ids, wins)
        _assert_same(got, solo, True, f"wave {wave}")
    s.stream_end()
    s.close()


def test_timed_mode(gm, ref):
    """Timed mode (plain launches with per-launch events, one lane): bit-identical, and the timed figures count."""
    import topay_b200 as tp
    plans, solo = ref
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=16)
    s.set_timed(True)
    got = _stream(s, plans[:6], "one_per_advance", True)
    st = s.stats()
    _assert_same(got, solo[:6], True, "timed")
    assert st["ms_eval"] > 0 and st["ms_lbfgs"] > 0
    s.close()


def test_row_reuse_and_a_full_store(gm):
    """64 store rows for 20 plans of 8 plus a 12-candidate plan of one repeated candidate: submits into a full store
    fail with TOO_LARGE and change nothing, taking a plan frees its rows, and the recycled rows reach the repeated
    plan out of order, so its tied candidates must go to the earliest one. Everything bit-identical to solo solves."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_TOO_LARGE, TopayError
    plans = _plans(20, seed0=7500)
    p0 = plans[0]
    tie = ([p0[0][1]] * 12, np.repeat(p0[1][1:2], 12, axis=0), np.repeat(p0[2][1:2], 12, axis=0))
    solo = _solos(gm, plans) + _solos(gm, [tie], max_cand=12)
    assert solo[-1]["win"][False][0] in (0, -1)
    s = tp.MomaTrajOpt(gm, max_cand=64, max_pieces=16, n_slots=16)
    s.stream_begin(use_gate=False)
    order = list(range(len(plans)))
    got, ids, wins = [None] * (len(plans) + 1), {}, {}
    refused, tie_at = 0, None
    for _ in range(MAX_ADVANCES):
        while order:
            try:
                ids[s.stream_submit(*plans[order[0]])] = order[0]
                order.pop(0)
            except TopayError as e:
                assert e.code == ERR_TOO_LARGE
                refused += 1
                break
        if not order and tie_at is None and len(ids) <= 3:
            tie_at = s.stream_submit(*tie)              # 12 rows, recycled from plans taken in different orders
            ids[tie_at] = len(plans)
        s.stream_advance(1)
        done = _poll(s, wins)
        for pid in sorted(done, reverse=True):          # take later plans first: the free rows come back shuffled
            _take(s, pid, got, ids, wins)
        if not order and tie_at is not None and not ids:
            break
    assert not ids and refused > 0
    s.stream_end()
    _assert_same(got, solo, False, "row reuse")
    s.close()


def test_per_plan_fields_with_the_gate(gm, small_scene):
    """Plans on three dense fields of different geometry (grids A-C of test_gpu_grid_geometry) and on the solver's own
    field, in one session with the gate: each bit-identical to a solo solve on its own field."""
    import topay_b200 as tp
    from topay_b200 import scenes
    from test_gpu_grid_geometry import GRIDS, _in_map_candidates, grid_spec
    fields, plans, which = [], [], []
    for k, name in enumerate(("A", "B", "C")):
        desc, lo, hi = grid_spec(name)
        f = tp.GridMap(desc)
        ms = desc.map_size
        pts, _ = scenes.cuboids_scene(90 + k, size_x=ms[0], size_y=ms[1], scale=np.sqrt(ms[0] * ms[1] / 400.0))
        f.regenerateMap(pts)
        fields.append(f)
        g = dict(lo=lo, hi=hi)
        for j in range(2):
            plans.append(_in_map_candidates(g, np.random.default_rng(800 + 10 * k + j), PLAN))
            which.append(f)
    plans += _plans(2, seed0=7700)
    which += [None, None]
    solo = []
    for f, p in zip(which, plans):
        solo += _solos(gm if f is None else f, [p])
    assert sum(e["win"][True][0] >= 0 for e in solo) >= 4
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=12)
    _assert_same(_stream(s, plans, "interleaved", True, fields=which), solo, True, "fields")
    s.close()
    for f in fields:
        f.close()


def test_session_on_a_slid_rog_ring():
    """A session on a ROG solver whose ring was slid so that its wrap runs through the candidates, with the gate:
    every plan bit-identical to a solo solve on the same ring; a dense field is refused."""
    import topay_b200 as tp
    from topay_b200 import scenes
    from topay_b200._lib import ERR_INVALID_ARG, TopayError
    from topay_b200.rog import ESDFMap
    from test_gpu_rog import OCC, UNK
    desc = tp.rog_desc(half_prob_map_size_i=(60, 40, 12), prob_resolution=0.1, esdf_resolution=0.2,
                       map_sliding_en=True)
    dev = ESDFMap(desc)
    odom = np.array([5.0, 3.3, 0.4])
    dev.mapSliding(odom)
    res, half = dev.resolution, (np.array(dev.map_size_i) - 1) // 2
    wrap = (half[:2] + 1) * res                                 # first world coordinate of ring cell 0
    lo = (np.array(dev.local_map_origin_i) - half) * res        # the local map
    hi = (np.array(dev.local_map_origin_i) + half + 1) * res
    pts, _ = scenes.cuboids_scene(5, size_x=11.0, size_y=7.0, scale=0.5)
    pts = pts.astype(np.float64) + np.array([odom[0], odom[1], 0.0])
    pts = pts[np.all((pts > lo + 0.01) & (pts < hi - 0.01), axis=1)]
    cells = np.unique(np.floor(pts / res).astype(np.int64), axis=0)
    dev.updateGridCounter((cells + 0.5) * res, UNK, OCC)
    dev.updateESDF3D(odom)
    rng = np.random.default_rng(9)
    plans = []
    for _ in range(4):
        paths = []
        while len(paths) < 6:
            a = wrap + rng.uniform([-1.8, -1.6], [-0.4, -0.4])
            b = wrap + rng.uniform([0.4, 0.4], [1.8, 1.6])
            if rng.random() < 0.5:
                a, b = b, a
            if 2.0 <= np.linalg.norm(b - a) <= 4.0:
                paths.append(scenes.scurve_candidate(rng, a, b, 8, 0.3))
        plans.append((paths, np.zeros((6, 10, 2)), np.zeros((6, 10, 2))))
    solo = _solos(dev, plans, max_cand=6)
    assert sum(e["res"]["status"].sum() for e in solo) >= 4
    s = tp.MomaTrajOpt(dev, max_cand=24, max_pieces=16)
    assert s.use_rog
    _assert_same(_stream(s, plans, "one_per_advance", True), solo, True, "rog")
    s.stream_begin()
    gm_other = tp.GridMap(tp.grid_desc())
    with pytest.raises(TopayError) as e:
        s.stream_submit(*plans[0], field=gm_other)
    assert e.value.code == ERR_INVALID_ARG
    s.stream_end()
    gm_other.close()
    s.close()
    dev.close()


def test_mode_discipline(gm, ref):
    """Batch calls are refused inside a session and stream calls outside one (NOT_READY); a plan is taken once, an
    unknown or unfinished plan is refused (INVALID_ARG); unbounded max_iterations is refused at stream_begin; after
    stream_end, a batch upload / run is bit-identical to a fresh solver."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_INVALID_ARG, ERR_NOT_READY, TopayError
    plans, solo = ref

    def refused(code, fn, *a, **kw):
        with pytest.raises(TopayError) as e:
            fn(*a, **kw)
        assert e.value.code == code, (fn, e.value)

    s = tp.MomaTrajOpt(gm, max_cand=4 * PLAN, max_pieces=16, n_slots=8)
    for fn, a in ((s.stream_advance, (1,)), (s.stream_poll, ()), (s.stream_take, (0,)), (s.stream_end, ()),
                  (s.stream_submit, plans[0])):
        refused(ERR_NOT_READY, fn, *a)
    s.upload(*plans[1])      # a batch upload in place before the session: dropped by stream_begin
    s.stream_begin(use_gate=True)
    refused(ERR_NOT_READY, s.stream_begin)
    pid = s.stream_submit(*plans[0])
    refused(ERR_INVALID_ARG, s.stream_take, pid)          # not finished
    refused(ERR_INVALID_ARG, s.stream_take, pid + 1)      # unknown
    refused(ERR_INVALID_ARG, s.stream_take, -1)
    prep = [tp.prepare_candidate(s.opt_param, s.moma_param, p, plans[0][1][0], plans[0][2][0], 16)
            for p in plans[0][0][:2]]
    batch_calls = [(s.upload, plans[0]), (s.run, ()), (s.download, ()), (s.download_candidate, (0,)),
                   (s.select, ()), (s.checkFeasibleBatch, ()), (s.assign_fields, ([gm, gm], [0] * PLAN)),
                   (s.set_plans, (None, 0)), (s.set_trace, (10,)), (s.set_timed, (True,)),
                   (s.evaluate, (1, [q["piece_num"] for q in prep], [q["head_pva"] for q in prep],
                                 [q["tail_pva"] for q in prep], [q["start_xy"] for q in prep],
                                 [q["end_xy"] for q in prep], [q["init_inner_xy"] for q in prep],
                                 [q["x0"] for q in prep]))]
    s._n = PLAN
    for fn, a in batch_calls:
        refused(ERR_NOT_READY, fn, *a)
    got, ids, wins = [None], {pid: 0}, {}
    _drain(s, got, ids, wins)
    _assert_same(got, solo[:1], True, "discipline")
    refused(ERR_INVALID_ARG, s.stream_take, pid)          # taken already
    s.stream_submit(*plans[2])                            # left unfinished: stream_end drops it
    s.stream_advance(1)
    s.stream_end()
    refused(ERR_NOT_READY, s.stream_poll)
    # batch mode again: bit-identical to a fresh solver on the same uploads
    fresh = tp.MomaTrajOpt(gm, max_cand=4 * PLAN, max_pieces=16, n_slots=8)
    for p in (plans[3], plans[4], plans[3]):
        for x in (s, fresh):
            x.upload(*p)
            x.run()
        a, b = s.download(), fresh.download()
        for k in RESULT_KEYS + ("best_by_duration", "best_by_cost"):
            assert np.array_equal(a[k], b[k]), k
    fresh.close()
    s.close()
    # unbounded iterations: a session could run forever
    opt = tp.opt_params_default()
    opt.s2_lbfgs.max_iterations = 0
    u = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16, opt_param=opt)
    refused(ERR_INVALID_ARG, u.stream_begin)
    u.close()
