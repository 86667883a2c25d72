"""First success + grace (topay_solver_set_plans): once a plan has a success, its candidates that need more than G
evaluations beyond the earliest success are cancelled, the way the planner's worker pool interrupts its workers a
grace period after the first success (planner.cpp:931-952), with the grace counted in evaluations.

Every expectation comes from an unbounded run of the same upload and the contract of include/topay_b200.h, applied on
the host by `contract()`: S_p = the fewest `evals` among the plan's successes (status 1 and, with the gate,
feasible_print); a candidate with evals <= S_p + G keeps its unbounded results, trace and gate metrics bit for bit,
every other one comes back cancelled (status 0, LBFGSERR_PLAN_GRACE, piece_num kept, everything else zero)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RESULT_KEYS = ("status", "lbfgs_code", "piece_num", "iters", "evals", "alm_rounds", "cost", "duration", "T", "coeff",
               "final_xy_err", "x")
ZEROED = ("iters", "evals", "alm_rounds", "cost", "duration", "T", "coeff", "final_xy_err", "x")
N_PLANS, PLAN = 50, 8
TRACE_CAP = 4000


def _reference_plans(n_plans, seed0=5000):
    """bench.latency_probe's plans: 8 candidates each, reference scale (int_K 12, 3-10 pieces)."""
    from topay_b200 import scenes
    return [scenes.short_candidates(PLAN, seed0 + p) for p in range(n_plans)]


def _cat(plans):
    return ([q for p in plans for q in p[0]], np.concatenate([p[1] for p in plans]),
            np.concatenate([p[2] for p in plans]))


def _offsets(plans):
    return np.cumsum([0] + [len(p[0]) for p in plans]).astype(np.int32)


def _solve(s, batch, off, grace, use_gate, fields=None, trace=True):
    """One run of `batch` on solver s: results, full gate metrics, per-plan winners and (optionally) traces."""
    s.upload(*batch)
    if fields is not None:
        s.assign_fields(fields, np.repeat(np.arange(len(fields)), np.diff(off)))
    s.set_plans(off, grace, use_gate)
    s.run()
    out = {"res": s.download(), "stats": s.stats()}
    out["gate"], _ = s.checkFeasibleBatch()
    out["gate"] = {k: v.copy() for k, v in out["gate"].items()}
    out["win"] = s.select(off, use_gate=bool(use_gate))
    out["win_status"] = s.select(off, use_gate=False)
    out["win_gate"] = s.select(off, use_gate=True)
    if trace:
        out["trace"] = [s.trace(c) for c in range(len(out["res"]["status"]))]
    return out


def contract(unb, off, grace, use_gate):
    """(kept mask, S per plan) of the contract, from an unbounded run."""
    r, fp = unb["res"], unb["gate"]["feasible_print"]
    keep, S = np.ones(len(r["status"]), bool), []
    for p in range(len(off) - 1):
        sl = slice(off[p], off[p + 1])
        ok = (r["status"][sl] == 1) & ((fp[sl] == 1) if use_gate else True)
        S.append(int(r["evals"][sl][ok].min()) if ok.any() else None)
        if S[-1] is not None:
            keep[sl] = r["evals"][sl] <= S[-1] + grace
    return keep, S


def _expected(unb, keep):
    import topay_b200 as tp
    res = {k: unb["res"][k].copy() for k in RESULT_KEYS}
    gone = ~keep
    res["status"][gone] = 0
    res["lbfgs_code"][gone] = tp.LBFGSERR_PLAN_GRACE
    for k in ZEROED:
        res[k][gone] = 0
    gate = {k: v.copy() for k, v in unb["gate"].items()}
    for v in gate.values():
        v[gone] = 0
    return res, gate


def _host_select(res, gate, off, use_gate):
    """planner.cpp:999-1010 on the expected survivors: the first success, replaced only by a strictly shorter one."""
    out = []
    for p in range(len(off) - 1):
        sl = slice(off[p], off[p + 1])
        ok = (res["status"][sl] == 1) & ((gate["feasible_print"][sl] == 1) if use_gate else True)
        idx = np.flatnonzero(ok)
        out.append(int(idx[np.argmin(res["duration"][sl][idx])]) if len(idx) else -1)
    return np.array(out)


def _assert_contract(got, unb, off, grace, use_gate, what, sl=slice(None), trace=True):
    """got (a run of the candidates `sl` of unb's upload, made of whole plans) against the contract."""
    full_off = unb["off"]
    keep, S = contract(unb, full_off, grace, use_gate)
    res, gate = _expected(unb, keep)
    for k in RESULT_KEYS:
        assert np.array_equal(got["res"][k], res[k][sl]), (what, k)
    for k, v in gate.items():
        assert np.array_equal(got["gate"][k], v[sl]), (what, "gate", k)
    n0 = 0 if sl.start is None else sl.start
    plans = [p for p in range(len(full_off) - 1) if full_off[p] >= n0 and full_off[p + 1] <= n0 + len(got["res"]["status"])]
    win = _host_select(res, gate, full_off, use_gate)[plans]
    assert np.array_equal(got["win"][0], win), (what, "select")
    assert np.array_equal(got["win_status"][0], _host_select(res, gate, full_off, False)[plans]), (what, "select status")
    unb_win = _host_select(unb["res"], unb["gate"], full_off, use_gate)[plans]
    assert np.all((unb_win >= 0) == (got["win"][0] >= 0)), (what, "a plan lost or gained its winner")
    if trace:
        for i, c in enumerate(range(n0, n0 + len(got["res"]["status"]))):
            exp = unb["trace"][c] if keep[c] else np.zeros((0, 4))
            assert np.array_equal(got["trace"][i], exp), (what, "trace", c)
    return keep[sl], S


@pytest.fixture(scope="module")
def gm(small_scene):
    import topay_b200 as tp
    g = tp.GridMap(small_scene["desc"], device=0)
    g.regenerateMap(small_scene["points"])
    yield g
    g.close()


@pytest.fixture(scope="module")
def ref(gm):
    """50 reference-scale plans of 8 through 400 slots (one lane, k_cand split while more than 384 are live), traced:
    the unbounded run every expectation is taken from, and a middle grace that cancels some candidates."""
    import topay_b200 as tp
    plans = _reference_plans(N_PLANS)
    batch, off = _cat(plans), _offsets(plans)
    s = tp.MomaTrajOpt(gm, max_cand=len(batch[0]), max_pieces=16)
    s.set_trace(TRACE_CAP)
    unb = _solve(s, batch, off, None, 0)
    unb["off"] = off
    over = []
    for use_gate in (0, 1):
        keep, S = contract(unb, off, 0, use_gate)
        for p, sp in enumerate(S):
            if sp is not None:
                e = unb["res"]["evals"][off[p]:off[p + 1]]
                over += list(e[e > sp] - sp)
    mid = int(np.median(over))
    print(f"unbounded: {int((unb['res']['status'] == 1).sum())} successes, {unb['stats']['ticks']} ticks, "
          f"max evals {unb['res']['evals'].max()}, middle grace {mid}")
    yield dict(s=s, plans=plans, batch=batch, off=off, unb=unb, mid=mid)
    s.close()


def test_off_means_off(ref):
    """A grace no candidate can exceed, set_plans(0) after an earlier setting, and the same upload after a grace run on
    the same solver: results, traces, gate metrics and per-plan winners bit-identical to the run without plans."""
    s, unb, off = ref["s"], ref["unb"], ref["off"]
    big = int(unb["res"]["evals"].max())
    runs = {"grace >= max evals": _solve(s, ref["batch"], off, big, 1)}
    s.set_plans(off, 0, 1)
    runs["set_plans(0) after a setting"] = _solve(s, ref["batch"], off, None, 0)
    _solve(s, ref["batch"], off, 0, 1, trace=False)
    s.set_plans(None)
    s.run()
    runs["same upload after a grace run"] = {"res": s.download(), "gate": s.checkFeasibleBatch()[0],
                                             "win_gate": s.select(off, True), "win_status": s.select(off, False),
                                             "trace": [s.trace(c) for c in range(off[-1])]}
    for what, got in runs.items():
        for k in RESULT_KEYS:
            assert np.array_equal(got["res"][k], unb["res"][k]), (what, k)
        for k, v in unb["gate"].items():
            assert np.array_equal(got["gate"][k], v), (what, "gate", k)
        for i in (0, 1):
            assert np.array_equal(got["win_status"][i], unb["win_status"][i]), (what, "select")
        for i in (0, 1):
            assert np.array_equal(got["win_gate"][i], unb["win_gate"][i]), (what, "gated select")
        assert np.array_equal(got["win_gate"][0], _host_select(unb["res"], unb["gate"], off, True)), what
        for c in range(off[-1]):
            assert np.array_equal(got["trace"][c], unb["trace"][c]), (what, "trace", c)


@pytest.mark.parametrize("use_gate", [0, 1], ids=["status", "gate"])
@pytest.mark.parametrize("which", ["zero", "middle"])
def test_contract_on_reference_plans(ref, which, use_gate):
    """Kept candidates bit-identical in every field, trace and gate entry; cancelled ones carry exactly the specified
    values; per-plan selection equals the host rule on the expected survivors; no plan loses its winner. The seeds
    include plans where grace cancels a candidate that would have won with a shorter duration, and (gated) plans whose
    first status-1 candidate fails printConstraintsSituations, the case that tells the two success tests apart."""
    s, unb, off = ref["s"], ref["unb"], ref["off"]
    grace = 0 if which == "zero" else ref["mid"]
    got = _solve(s, ref["batch"], off, grace, use_gate)
    keep, S = _assert_contract(got, unb, off, grace, use_gate, (which, use_gate))
    r, fp = unb["res"], unb["gate"]["feasible_print"]
    over = sum(int((r["evals"][off[p]:off[p + 1]] > S[p]).sum()) for p in range(N_PLANS) if S[p] is not None)
    assert 0 < (~keep).sum(), "grace cancelled nothing"
    if which == "middle":
        assert (~keep).sum() < over, "the middle grace cancelled every candidate past the first success"
    ok = (r["status"] == 1) & ((fp == 1) if use_gate else True)
    lost_better = []
    for p in range(N_PLANS):
        if S[p] is None:
            continue
        c = np.arange(off[p], off[p + 1])
        first = c[ok[c] & (r["evals"][c] == S[p])][0]
        if (ok[c] & ~keep[c] & (r["duration"][c] < r["duration"][first])).any():
            lost_better.append(p)
    print(f"grace {grace}, gate {use_gate}: {(~keep).sum()} of {len(keep)} cancelled, "
          f"plans that lost a shorter success: {len(lost_better)}, ticks {got['stats']['ticks']} "
          f"(unbounded {unb['stats']['ticks']})")
    if which == "zero":
        assert lost_better, "no plan cancels a candidate that would have succeeded with a shorter duration"
    if use_gate:
        first_fails = []
        for p in range(N_PLANS):
            c = np.arange(off[p], off[p + 1])
            c = c[r["status"][c] == 1]
            if len(c) and fp[c[np.argmin(r["evals"][c])]] == 0:
                first_fails.append(p)
        print(f"plans whose earliest status-1 candidate fails the gate: {first_fails}")
        assert first_fails, "no plan whose earliest status-1 candidate fails the gate"


def test_independent_of_scheduling(ref, gm, monkeypatch):
    """The same gated grace batch through all 400 slots, 8 and 3 slots (plans queued behind running ones), two lanes,
    timed mode (k_cand split throughout) and the 400-slot lane that starts split: bit-identical to the contract."""
    import topay_b200 as tp
    unb, off, grace = ref["unb"], ref["off"], ref["mid"]
    n = int(off[-1])
    s = ref["s"]
    got = _solve(s, ref["batch"], off, grace, 1)
    _assert_contract(got, unb, off, grace, 1, "400 slots")
    assert got["stats"]["eval_launches"] == got["stats"]["ticks"]
    s.set_timed(True)
    got = _solve(s, ref["batch"], off, grace, 1)
    s.set_timed(False)
    assert got["stats"]["ms_adj"] > 0 and got["stats"]["ms_lbfgs"] > 0
    _assert_contract(got, unb, off, grace, 1, "timed")
    monkeypatch.setenv("TOPAY_LANE_MIN_SLOTS", "2")
    two = tp.MomaTrajOpt(gm, max_cand=n, max_pieces=16)
    two.set_trace(TRACE_CAP)
    got = _solve(two, ref["batch"], off, grace, 1)
    assert got["stats"]["eval_launches"] == 2 * got["stats"]["ticks"], got["stats"]
    _assert_contract(got, unb, off, grace, 1, "two lanes")
    two.close()
    monkeypatch.delenv("TOPAY_LANE_MIN_SLOTS")
    k = 12      # the first 12 plans through few slots: plans wait in the queue behind running ones
    sub_plans = ref["plans"][:k]
    for ns in (8, 3):
        few = tp.MomaTrajOpt(gm, max_cand=k * PLAN, max_pieces=16, n_slots=ns)
        few.set_trace(TRACE_CAP)
        got = _solve(few, _cat(sub_plans), _offsets(sub_plans), grace, 1)
        _assert_contract(got, unb, off, grace, 1, f"{ns} slots", sl=slice(0, k * PLAN))
        few.close()


def test_independent_of_scheduling_in_a_scenario_sweep():
    """Eight scenarios with their own fields, two plans of 8 each, in one upload (assign_fields: the MULTI penalty
    kernel and a gate that reads every candidate's own field): gated grace through all slots and through 16 slots,
    both bit-identical to the contract applied to the unbounded run of the same upload."""
    import topay_b200 as tp
    from topay_b200 import scenes
    fields, plans = [], []
    for sc in range(8):
        g = tp.GridMap(tp.grid_desc())
        g.regenerateMap(scenes.tables_scene(90 + sc)[0] if sc % 2 == 0 else scenes.cuboids_scene(90 + sc)[0])
        fields.append(g)
        plans += _reference_plans(2, 7000 + 10 * sc)
    batch, off = _cat(plans), _offsets(plans)
    field_of_plan = [fields[p // 2] for p in range(len(plans))]
    n = int(off[-1])
    s = tp.MomaTrajOpt(fields[0], max_cand=n, max_pieces=16)
    s.set_trace(TRACE_CAP)
    unb = _solve(s, batch, off, None, 0, fields=field_of_plan)
    unb["off"] = off
    keep, S = contract(unb, off, 0, 1)
    few = tp.MomaTrajOpt(fields[0], max_cand=n, max_pieces=16, n_slots=16)
    few.set_trace(TRACE_CAP)
    for what, solver in (("all slots", s), ("16 slots", few)):
        got = _solve(solver, batch, off, 0, 1, fields=field_of_plan)
        _assert_contract(got, unb, off, 0, 1, what)
    assert (~keep).any()
    s.close()
    few.close()
    for g in fields:
        g.close()


@pytest.mark.parametrize("use_gate", [0, 1], ids=["status", "gate"])
def test_the_tail_is_cut(ref, gm, use_gate):
    """One plan with every candidate in flight whose slowest candidate needs more than S + G + 32 evaluations: the run
    ends after at most ceil((S + G + 1) / 16) batches of 16 ticks plus one (plus two with the gate, which is applied
    between batches), and before the unbounded run's end. Counted in ticks, not timed."""
    import topay_b200 as tp
    unb, off = ref["unb"], ref["off"]
    grace = 0
    keep, S = contract(unb, off, grace, use_gate)
    gaps = [(int(unb["res"]["evals"][off[p]:off[p + 1]].max()) - S[p], p) for p in range(N_PLANS) if S[p] is not None]
    gap, p = max(gaps)
    assert gap > grace + 32, gaps
    plan = ref["plans"][p]
    one = tp.MomaTrajOpt(gm, max_cand=PLAN, max_pieces=16)
    poff = np.array([0, PLAN], np.int32)
    one.upload(*plan)
    one.set_plans(None)
    one.run()
    ticks_unb = one.stats()["ticks"]
    one.set_plans(poff, grace, use_gate)
    one.run()
    ticks = one.stats()["ticks"]
    res = one.download()
    one.close()
    sl = slice(off[p], off[p + 1])
    assert np.array_equal(res["evals"], np.where(keep[sl], unb["res"]["evals"][sl], 0))
    bound = -(-(S[p] + grace + 1) // 16) * 16 + (32 if use_gate else 16)
    print(f"plan {p}: S {S[p]}, max evals {S[p] + gap}, ticks {ticks} (bound {bound}, unbounded {ticks_unb})")
    assert ticks < ticks_unb and ticks <= bound, (ticks, bound, ticks_unb)


def test_headline_shape_in_two_split_lanes(gm):
    """776 candidates of 64 pieces x K = 32 as three plans through 776 slots (two split lanes): the contract holds."""
    import topay_b200 as tp
    from topay_b200 import scenes
    n = 776
    opt = tp.opt_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    paths, bv, ba = scenes.synthetic_batch(n, 1234)
    off = np.array([0, 259, 518, n], np.int32)
    s = tp.MomaTrajOpt(gm, max_cand=n, max_pieces=64, opt_param=opt, n_slots=n)
    unb = _solve(s, (paths, bv, ba), off, None, 0, trace=False)
    unb["off"] = off
    grace = 100
    got = _solve(s, (paths, bv, ba), off, grace, 0, trace=False)
    assert got["stats"]["eval_launches"] == 2 * got["stats"]["ticks"], got["stats"]
    keep, _ = _assert_contract(got, unb, off, grace, 0, "headline", trace=False)
    print(f"headline: {(~keep).sum()} of {n} cancelled, ticks {got['stats']['ticks']} (unbounded {unb['stats']['ticks']})")
    assert (~keep).any() and got["stats"]["ticks"] < unb["stats"]["ticks"]
    s.close()


def test_gated_grace_on_a_slid_rog_ring():
    """ROG mode: a gated grace batch of two plans on a slid ring; the in-solve gate reads the ring. The contract holds.
    On this ring every status-1 candidate fails printConstraintsSituations, so the gated rule cancels nothing here,
    while a success published on status alone would cancel candidates."""
    import topay_b200 as tp
    from topay_b200 import scenes
    from topay_b200.rog import ESDFMap
    from test_gpu_rog import OCC, UNK
    desc = tp.rog_desc(half_prob_map_size_i=(60, 40, 12), prob_resolution=0.1, esdf_resolution=0.2,
                       map_sliding_en=True)
    dev = ESDFMap(desc)
    res = dev.resolution
    odom = np.array([5.0, 3.3, 0.4])
    dev.mapSliding(odom)
    half = (np.array(dev.map_size_i) - 1) // 2
    wrap = (half[:2] + 1) * res                                 # first world coordinate of ring cell 0
    lo = (np.array(dev.local_map_origin_i) - half) * res        # the local map
    hi = (np.array(dev.local_map_origin_i) + half + 1) * res
    pts, _ = scenes.cuboids_scene(5, size_x=11.0, size_y=7.0, scale=0.5)
    pts = pts.astype(np.float64) + np.array([odom[0], odom[1], 0.0])
    pts = pts[np.all((pts > lo + 0.01) & (pts < hi - 0.01), axis=1)]
    centres = (np.unique(np.floor(pts / res).astype(np.int64), axis=0) + 0.5) * res
    dev.updateGridCounter(centres, UNK, OCC)
    dev.updateESDF3D(odom)
    rng = np.random.default_rng(9)
    paths = []
    while len(paths) < 16:
        a = wrap + rng.uniform([-1.8, -1.6], [-0.4, -0.4])
        b = wrap + rng.uniform([0.4, 0.4], [1.8, 1.6])
        if 2.0 <= np.linalg.norm(b - a) <= 4.0:
            paths.append(scenes.scurve_candidate(rng, a, b, 8, 0.3))
    batch = (paths, np.zeros((16, 10, 2)), np.zeros((16, 10, 2)))
    off = np.array([0, 8, 16], np.int32)
    s = tp.MomaTrajOpt(dev, max_cand=16, max_pieces=16)
    assert s.use_rog
    s.set_trace(TRACE_CAP)
    unb = _solve(s, batch, off, None, 0)
    unb["off"] = off
    got = _solve(s, batch, off, 0, 1)
    keep, S = _assert_contract(got, unb, off, 0, 1, "rog")
    print(f"ROG ring: S {S}, {(~keep).sum()} of 16 cancelled")
    assert (unb["res"]["status"] == 1).any()      # the in-solve gate ran on the ring
    s.close()
    dev.close()


def test_set_plans_arguments_and_upload_size():
    """Malformed offsets, a negative grace and more plans than candidates are INVALID_ARG; a run after an upload of
    another size is NOT_READY with its own error text (the style of test_gpu_call_contract)."""
    from topay_b200 import _lib
    from topay_b200 import GridMap, MomaTrajOpt
    from topay_b200 import scenes
    from test_gpu_call_contract import PRIMED, _prime
    g = GridMap()
    g.regenerateMap(scenes.cuboids_scene(42)[0])
    s = MomaTrajOpt(g, max_cand=8, max_pieces=16)
    l = _lib.lib()
    paths, bv, ba = scenes.short_candidates(8, 5000)
    s.upload(paths, bv, ba)

    def sp(off, grace=0):
        off = np.ascontiguousarray(off, dtype=np.int32)
        return l.topay_solver_set_plans(s.h, len(off) - 1, off.ctypes.data_as(C.POINTER(C.c_int32)), 1, grace)

    for bad in ([1, 8], [0, 7], [0, 5, 3, 8], [0, 9], [0, 4, 9]):
        assert sp(bad) == _lib.ERR_INVALID_ARG, bad
    assert sp([0, 8], grace=-1) == _lib.ERR_INVALID_ARG
    assert sp([0] * 9 + [8]) == _lib.ERR_INVALID_ARG     # nine plans (some empty) of eight candidates
    assert l.topay_solver_set_plans(s.h, -1, None, 0, 0) == _lib.ERR_INVALID_ARG
    assert sp([0, 4, 8], grace=5) == _lib.OK
    assert sp(list(range(9))) == _lib.OK           # eight plans of one
    s.upload(paths[:4], bv[:4], ba[:4])
    _prime(g.h)
    assert l.topay_solver_run(s.h) == _lib.ERR_NOT_READY
    assert l.topay_last_error().decode() != PRIMED
    s.set_plans(None)                               # off: any size runs
    s.run()
    assert s.download()["status"].shape == (4,)
    s.close()
    g.close()
