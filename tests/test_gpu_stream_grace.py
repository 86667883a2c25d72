"""First success + grace and stopped plans in streaming sessions (topay_solver_stream_set_grace, _stream_stop).

A plan streamed with grace G must be bit-identical to the same plan solved alone through the batch API on a fresh upload
with set_plans(1, {0, n}, use_gate, G): every result field, every gate metric and both winners. Those solo solves are
checked against the contract itself by test_gpu_plan_grace.py, so they are the expectations here. A stopped plan keeps
the candidates that finished before the stop (under its grace contract) bit for bit and cancels the rest; the other
plans of the session do not change. Every loop that waits for plans is bounded."""
import numpy as np
import pytest

from test_gpu_stream import MAX_ADVANCES, PLAN, RESULT_KEYS, _drain, _plans, _poll, _stream, _take

pytestmark = pytest.mark.gpu

ZEROED = ("iters", "evals", "alm_rounds", "cost", "duration", "T", "coeff", "final_xy_err", "x")


def _solo(solver, plan, grace, use_gate):
    """The plan alone on a fresh upload with set_plans(1, {0, n}, use_gate, grace) (None: unbounded): results, gate
    metrics, winners with and without the gate."""
    solver.upload(*plan)
    solver.set_plans(None, grace, use_gate)
    solver.run()
    res = {k: v.copy() for k, v in solver.download().items() if k in RESULT_KEYS}
    gate, _ = solver.checkFeasibleBatch()
    win = {g: tuple(int(v[0]) for v in solver.select(None, use_gate=g)) for g in (False, True)}
    return dict(res=res, gate={k: v.copy() for k, v in gate.items()}, win=win)


def _first_success(e, use_gate):
    """S of a solo result: the fewest evals among its successes (None: no success)."""
    ok = (e["res"]["status"] == 1) & ((e["gate"]["feasible_print"] == 1) if use_gate else True)
    return int(e["res"]["evals"][ok].min()) if ok.any() else None


def _assert_same(got, exp, use_gate, what):
    for k in RESULT_KEYS:
        assert np.array_equal(got["res"][k], exp["res"][k]), (what, k)
    for k, v in exp["gate"].items():
        assert np.array_equal(got["gate"][k], v), (what, "gate", k)
    assert got["win"] == exp["win"][use_gate], (what, "winners", got["win"], exp["win"][use_gate])


def _assert_all_same(got, solo, use_gate, what):
    for p, (g, e) in enumerate(zip(got, solo)):
        _assert_same(g, e, use_gate, (what, p))


class _Graced:
    """A solver whose stream_begin also sets the session's grace, so that test_gpu_stream's schedules drive it."""

    def __init__(self, s, grace):
        self.s, self.grace = s, grace

    def __getattr__(self, k):
        return getattr(self.s, k)

    def stream_begin(self, use_gate=False):
        self.s.stream_begin(use_gate=use_gate, grace_evals=self.grace)


def _refused(code, fn, *a):
    from topay_b200._lib import TopayError
    with pytest.raises(TopayError) as e:
        fn(*a)
    assert e.value.code == code, (fn, e.value)


@pytest.fixture(scope="module")
def gm(small_scene):
    import topay_b200 as tp
    g = tp.GridMap(small_scene["desc"], device=0)
    g.regenerateMap(small_scene["points"])
    yield g
    g.close()


@pytest.fixture(scope="module")
def ref(gm):
    """12 reference-scale plans of 8: the first ten of test_gpu_plan_grace's seeds and two of its plans whose earliest
    status-1 candidate fails the gate. Their solo solves unbounded and at G = 0 and a middle G, with and without the
    gate, keyed (G, use_gate)."""
    import topay_b200 as tp
    pool = _plans(50, seed0=5000)
    s = tp.MomaTrajOpt(gm, max_cand=len(pool) * PLAN, max_pieces=16)
    s.upload([q for p in pool for q in p[0]], np.concatenate([p[1] for p in pool]), np.concatenate([p[2] for p in pool]))
    s.run()
    r = s.download()
    fp = s.checkFeasibleBatch()[0]["feasible_print"].copy()
    s.close()
    first_fails = []
    for p in range(len(pool)):
        c = np.arange(p * PLAN, (p + 1) * PLAN)
        c = c[r["status"][c] == 1]
        if len(c) and fp[c[np.argmin(r["evals"][c])]] == 0:
            first_fails.append(p)
    assert first_fails, "no plan whose earliest status-1 candidate fails the gate"
    chosen = list(range(10)) + [p for p in first_fails if p >= 10][:2]
    plans = [pool[p] for p in chosen]
    one = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16)
    unb = [_solo(one, p, None, 0) for p in plans]
    over = []
    for use_gate in (False, True):
        for e in unb:
            S = _first_success(e, use_gate)
            if S is not None:
                ev = e["res"]["evals"]
                over += list(ev[ev > S] - S)
    mid = int(np.median(over))
    solo = {(None, g): unb for g in (False, True)}
    for G in (0, mid):
        for g in (False, True):
            solo[(G, g)] = [_solo(one, p, G, int(g)) for p in plans]
    one.close()
    print(f"plans {chosen}, middle grace {mid}")
    return dict(plans=plans, solo=solo, mid=mid, first_fails=[chosen.index(p) for p in chosen if p in first_fails])


@pytest.mark.parametrize("schedule", ["upfront", "interleaved"])
@pytest.mark.parametrize("use_gate", [False, True], ids=["status", "gate"])
@pytest.mark.parametrize("which", ["zero", "middle"])
def test_contract(gm, ref, which, use_gate, schedule):
    """Plans streamed with G = 0 and a middle G through 8 slots (plans wait in the queue behind running ones): every
    plan bit-identical to its solo solve with that grace. Some plans have candidates the grace rule cancels, and with
    the gate some plan's earliest status-1 candidate fails it, so publishing on status alone would differ."""
    import topay_b200 as tp
    plans, G = ref["plans"], 0 if which == "zero" else ref["mid"]
    exp = ref["solo"][(G, use_gate)]
    assert any((e["res"]["lbfgs_code"] == tp.LBFGSERR_PLAN_GRACE).any() for e in exp), "grace cancelled nothing"
    if use_gate:
        assert ref["first_fails"]
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=8)
    _assert_all_same(_stream(_Graced(s, G), plans, schedule, use_gate), exp, use_gate, (which, schedule))
    s.close()


@pytest.mark.parametrize("pool", ["3 slots", "all slots", "two lanes", "timed"])
def test_independent_of_scheduling(gm, ref, pool):
    """The same gated grace stream through 3 slots, all slots, a 512-slot pool in two lanes and timed mode: every plan
    bit-identical to its solo solve."""
    import topay_b200 as tp
    plans, G = ref["plans"], ref["mid"]
    exp = ref["solo"][(G, True)]
    n_slots = {"3 slots": 3, "all slots": None, "two lanes": 512, "timed": 16}[pool]
    s = tp.MomaTrajOpt(gm, max_cand=512 if pool == "two lanes" else len(plans) * PLAN, max_pieces=16, n_slots=n_slots)
    if pool == "timed":
        s.set_timed(True)
        plans, exp = plans[:6], exp[:6]
    got = _stream(_Graced(s, G), plans, "one_per_advance" if pool == "timed" else "interleaved", True)
    st = s.stats()
    _assert_all_same(got, exp, True, pool)
    if pool == "two lanes":
        assert st["eval_launches"] == 2 * st["ticks"], st
    if pool == "timed":
        assert st["ms_lbfgs"] > 0
    s.close()


def test_plan_id_reuse(gm, ref):
    """A plan with an early success is taken, and a plan whose successes come later reuses its id and its store rows
    (an 8-row store): the new plan matches its own solo solve, so the earlier plan's first success does not carry
    over."""
    import topay_b200 as tp
    plans, unb, exp = ref["plans"], ref["solo"][(None, False)], ref["solo"][(0, False)]
    S = [_first_success(e, False) for e in unb]
    a = min((v, p) for p, v in enumerate(S) if v is not None)[1]
    # b: a candidate kept at G = 0 runs past a's first success, which the id's old bound would cancel
    b = next(p for p in range(len(plans))
             if p != a and (exp[p]["res"]["evals"] > S[a]).any() and (S[p] is None or S[p] > S[a]))
    s = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16)
    s.stream_begin(use_gate=False, grace_evals=0)
    got, ids, wins = [None, None], {}, {}
    pa = s.stream_submit(*plans[a])
    ids[pa] = 0
    _drain(s, got, ids, wins)
    pb = s.stream_submit(*plans[b])
    assert pb == pa
    ids[pb] = 1
    _drain(s, got, ids, wins)
    s.stream_end()
    s.close()
    _assert_all_same(got, [exp[a], exp[b]], False, "reuse")


def test_grace_turned_off(gm, ref):
    """Grace on, plans finish, grace off (-1) with the finished plans not taken yet, then the same plans again: the
    first wave matches the G = 0 solo solves, the second the unbounded ones. set_grace is refused while a plan is live
    (NOT_READY) and outside a session (NOT_READY); -2 is INVALID_ARG."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_INVALID_ARG, ERR_NOT_READY
    plans = ref["plans"]
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16, n_slots=8)
    _refused(ERR_NOT_READY, s.stream_set_grace, 0)
    s.stream_begin(use_gate=True, grace_evals=0)
    for wave, key in enumerate(((0, True), (None, True))):
        got, ids, wins = [None] * len(plans), {}, {}
        for i, p in enumerate(plans):
            ids[s.stream_submit(*p)] = i
        _refused(ERR_NOT_READY, s.stream_set_grace, -1)
        _refused(ERR_INVALID_ARG, s.stream_set_grace, -2)
        _drain(s, got, ids, wins, take=False)
        if wave == 0:
            s.stream_set_grace(None)        # allowed: every plan has finished, none is taken yet
        for pid in list(wins):
            _take(s, pid, got, ids, wins)
        _assert_all_same(got, ref["solo"][key], True, f"wave {wave}")
    s.stream_end()
    _refused(ERR_NOT_READY, s.stream_set_grace, -1)
    s.close()


def _cancelled(got, unb):
    """got (a taken plan) carries the cancelled values at every candidate."""
    import topay_b200 as tp
    r = got["res"]
    return bool((r["status"] == 0).all() and (r["lbfgs_code"] == tp.LBFGSERR_PLAN_GRACE).all()
                and np.array_equal(r["piece_num"], unb["res"]["piece_num"])
                and all(not r[k].any() for k in ZEROED) and all(not v.any() for v in got["gate"].values()))


def _host_win(got, use_gate):
    """planner.cpp:999-1010 on a taken plan: the first success, replaced only by a strictly smaller duration / cost."""
    r = got["res"]
    ok = np.flatnonzero((r["status"] == 1) & ((got["gate"]["feasible_print"] == 1) if use_gate else True))
    if not len(ok):
        return (-1, -1)
    return int(ok[np.argmin(r["duration"][ok])]), int(ok[np.argmin(r["cost"][ok])])


@pytest.mark.parametrize("grace", ["off", "middle"])
def test_stop(gm, ref, grace):
    """Every candidate in a slot. One plan is stopped before any advance: all its candidates come back cancelled, with
    no winner, reported once. One is stopped mid-run: it is reported by the next advance, every candidate is either
    bit-identical to its unbounded solo result or cancelled, the candidates that finished a batch before the stop and
    are kept by the grace contract are kept, and the winners follow planner.cpp:999-1010 over the kept ones. A stop of
    a finished plan changes nothing, an unknown or taken id is INVALID_ARG, a stop outside a session NOT_READY. Every
    other plan is bit-identical to its solo solve. Grace off (the first stop turns the plans' bounds on) with the
    status test, and a middle grace with the gate."""
    import topay_b200 as tp
    from topay_b200._lib import ERR_INVALID_ARG, ERR_NOT_READY
    plans = ref["plans"]
    G, use_gate = (None, False) if grace == "off" else (ref["mid"], True)
    unb, exp = ref["solo"][(None, use_gate)], ref["solo"][(G, use_gate)]

    def live_until(p):      # evaluations until the plan's last candidate ends in its solo run (plus the grace step)
        S = _first_success(unb[p], use_gate)
        ev = unb[p]["res"]["evals"]
        return int(ev.max() if S is None or G is None else np.minimum(ev, S + G + 1).max())

    early = 0
    mid = max(range(1, len(plans)), key=lambda p: live_until(p) - int(unb[p]["res"]["evals"].min()))
    b = max(2, -(-int(unb[mid]["res"]["evals"].min()) // 16) + 1)     # advances before the stop
    assert 16 * b + 32 < live_until(mid), (b, live_until(mid))
    s = tp.MomaTrajOpt(gm, max_cand=len(plans) * PLAN, max_pieces=16)
    _refused(ERR_NOT_READY, s.stream_stop, 0)
    s.stream_begin(use_gate=use_gate, grace_evals=G)
    got, ids, wins = [None] * len(plans), {}, {}
    pid = [s.stream_submit(*p) for p in plans]
    ids.update({q: i for i, q in enumerate(pid)})
    s.stream_stop(pid[early])
    stopped_done = False
    for k in range(1, MAX_ADVANCES):
        live = s.stream_advance(1)
        reported = _poll(s, wins)
        if k == b:
            assert pid[mid] not in wins, "the plan finished before its stop"
            s.stream_stop(pid[mid])
        if k == b + 1:
            assert pid[mid] in wins, "a stopped plan whose candidates are all in slots was not reported"
        for q in reported:
            if not stopped_done and q not in (pid[early], pid[mid]):
                s.stream_stop(q)                # finished, not taken: nothing changes
                stopped_done = True
            _take(s, q, got, ids, wins)
        if live == 0 and not ids:
            break
    assert not ids and stopped_done
    _refused(ERR_INVALID_ARG, s.stream_stop, pid[mid])          # taken
    _refused(ERR_INVALID_ARG, s.stream_stop, len(plans) * PLAN - 1)   # never handed out
    _refused(ERR_INVALID_ARG, s.stream_stop, -1)
    s.stream_end()
    _refused(ERR_NOT_READY, s.stream_stop, pid[early])
    s.close()
    assert _cancelled(got[early], unb[early]) and got[early]["win"] == (-1, -1), "plan stopped before any advance"
    g, u = got[mid], unb[mid]
    kept = g["res"]["lbfgs_code"] != tp.LBFGSERR_PLAN_GRACE
    for c in range(PLAN):
        one = {"res": {k: v[c] for k, v in g["res"].items()}, "gate": {k: v[c] for k, v in g["gate"].items()}}
        if kept[c]:
            for k in RESULT_KEYS:
                assert np.array_equal(one["res"][k], u["res"][k][c]), ("mid-run stop", c, k)
            for k, v in u["gate"].items():
                assert np.array_equal(one["gate"][k], v[c]), ("mid-run stop", c, "gate", k)
        else:
            assert one["res"]["status"] == 0 and one["res"]["piece_num"] == u["res"]["piece_num"][c]
            assert all(not np.any(one["res"][k]) for k in ZEROED) and all(not np.any(v) for v in one["gate"].values())
    contract_kept = exp[mid]["res"]["lbfgs_code"] != tp.LBFGSERR_PLAN_GRACE
    finished = u["res"]["evals"] <= 16 * (b - 1)
    assert (finished & contract_kept).any() and (~kept).any()
    assert kept[finished & contract_kept].all(), "a candidate that finished before the stop was cancelled"
    assert g["win"] == _host_win(g, use_gate), ("mid-run stop winners", g["win"])
    others = [p for p in range(len(plans)) if p not in (early, mid)]
    _assert_all_same([got[p] for p in others], [exp[p] for p in others], use_gate, "other plans")
    print(f"grace {grace}: stopped after {b} advances, {int(kept.sum())} of {PLAN} kept, winners {g['win']}")


@pytest.mark.parametrize("use_gate", [False, True], ids=["status", "gate"])
def test_the_tail_is_cut(gm, ref, use_gate):
    """G = 0, every candidate in a slot, a plan whose slowest candidate needs far more than S + G evaluations: the plan
    is reported within ceil((S + G + 1) / 16) + 1 advances of one batch (+ 3 with the gate, applied between batches),
    sooner than its slowest candidate would end, and matches its solo solve."""
    import topay_b200 as tp
    plans, unb, exp = ref["plans"], ref["solo"][(None, use_gate)], ref["solo"][(0, use_gate)]
    gaps = [(int(e["res"]["evals"].max()) - S, p) for p, e in enumerate(unb)
            if (S := _first_success(e, use_gate)) is not None]
    gap, p = max(gaps)
    S = _first_success(unb[p], use_gate)
    assert gap > 64, gaps
    s = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16)
    s.stream_begin(use_gate=use_gate, grace_evals=0)
    got, ids, wins = [None], {s.stream_submit(*plans[p]): 0}, {}
    for k in range(1, MAX_ADVANCES):
        s.stream_advance(1)
        if _poll(s, wins):
            break
    _take(s, next(iter(wins)), got, ids, wins)
    s.stream_end()
    s.close()
    bound = -(-(S + 1) // 16) + (3 if use_gate else 1)
    print(f"plan {p}: S {S}, max evals {S + gap}, reported after {k} advances (bound {bound})")
    assert k <= bound and 16 * k < S + gap, (k, bound, S + gap)
    _assert_same(got[0], exp[p], use_gate, "tail")


def test_gated_grace_session_on_a_slid_rog_ring():
    """A gated G = 0 session on a ROG solver whose slid ring wraps through the candidates: the in-session gate reads the
    ring, and every plan is bit-identical to its solo solve on the same ring."""
    import topay_b200 as tp
    from topay_b200 import scenes
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
    one = tp.MomaTrajOpt(dev, max_cand=6, max_pieces=16)
    solo = [_solo(one, p, 0, 1) for p in plans]
    one.close()
    assert sum(e["res"]["status"].sum() for e in solo) >= 4
    s = tp.MomaTrajOpt(dev, max_cand=24, max_pieces=16)
    assert s.use_rog
    _assert_all_same(_stream(_Graced(s, 0), plans, "one_per_advance", True), solo, True, "rog")
    s.close()
    dev.close()
