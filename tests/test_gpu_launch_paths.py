"""The launch configurations the solver chooses at run time from the live-slot count, the lane threshold and the timed
switch, at the pool sizes that reach them (topay_b200/csrc/solver.cu, enqueue_lane / topay_solver_run):

* fused: up to TP_FUSE_MAX_SLOTS (444) live slots per lane a tick runs k_cand as one launch of all three halves;
* split: above that, and always in timed mode, k_cand runs as three launches (adjoint, L-BFGS, generate) that hand
  the candidate's state over through global memory, the L-BFGS launch with a ring of its own depth;
* two lanes: from 512 seeded slots on (TOPAY_LANE_MIN_SLOTS) the slots run as two parallel chains;
* MULTI: a scenario sweep's k_penalty reads each candidate's own field.

None of these may change a result: every test compares bit for bit with a configuration the rest of the suite pins to
the oracle (a fused, single-lane, graph-mode solve), and asserts from the launch counts that it took the path it
claims. A lane-batch of 16 ticks is k_list_roll plus 16 x (3 evaluation kernels + k_cand): 65 launches fused, 97
split; a run adds k_slot_init and the first generate launch."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RESULT_KEYS = ("status", "lbfgs_code", "evals", "iters", "alm_rounds", "cost", "T", "coeff", "x", "final_xy_err")
FUSED, SPLIT = 1 + 16 * 4, 1 + 16 * 6


@pytest.fixture(scope="module")
def gpu_scene(small_scene):
    import topay_b200 as tp
    gm = tp.GridMap(small_scene["desc"], device=0)
    gm.regenerateMap(small_scene["points"])
    yield gm
    gm.close()


def _headline_opt():
    import topay_b200 as tp
    opt = tp.opt_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    return opt


def _split_batches(st, lanes):
    """Lane-batches of the last run that ran k_cand split, from its launch counts."""
    assert st["ticks"] % 16 == 0 and st["eval_launches"] == lanes * st["ticks"], st
    extra = st["kernel_launches"] - 2 - FUSED * lanes * st["ticks"] // 16
    assert extra >= 0 and extra % (SPLIT - FUSED) == 0, st
    return extra // (SPLIT - FUSED)


def _assert_same_results(a, b, what):
    for k in RESULT_KEYS:
        assert np.array_equal(a[k], b[k]), (what, k)


def _assert_same_winner(a, b, what):
    assert (a is None) == (b is None), what
    if a is not None:
        for k, v in a.items():
            assert np.array_equal(v, b[k]), (what, k)


def test_split_then_fused_within_one_run(gpu_scene, monkeypatch):
    """400 short candidates through 400 slots in one lane: the run starts split (a grid of 512 live slots) and turns
    fused once at most 384 are left. Bit-identical to the same batch through 32 slots (fused throughout), per-plan
    winners and gate verdicts included."""
    import topay_b200 as tp
    from topay_b200 import scenes
    monkeypatch.setenv("TOPAY_LANE_MIN_SLOTS", "0")
    n = 400
    paths, bv, ba = scenes.short_candidates(n, 21)
    plans = [(paths[i:i + 8], bv[i:i + 8], ba[i:i + 8]) for i in range(0, n, 8)]
    res, win, gate, split = {}, {}, {}, {}
    for ns in (n, 32):
        s = tp.MomaTrajOpt(gpu_scene, max_cand=n, max_pieces=16, n_slots=ns)
        res[ns] = s.optimizeTrajBatch(paths, bv, ba)
        st = s.stats()
        split[ns] = _split_batches(st, 1)
        if ns == n:
            assert 0 < split[ns] < st["ticks"] // 16, (split[ns], st["ticks"])
        win[ns] = s.planWinners(plans, use_gate=True)
        gate[ns] = {k: v.copy() for k, v in s.constraints.items()}
        s.close()
    print(f"split lane-batches: {split}")
    assert split[32] == 0
    _assert_same_results(res[n], res[32], "400 vs 32 slots")
    assert (res[n]["status"] == 1).any()
    for i, (a, b) in enumerate(zip(win[32], win[n])):
        _assert_same_winner(a, b, i)
    assert any(w is not None for w in win[n])
    for k in ("feasible", "feasible_print"):
        assert np.array_equal(gate[n][k], gate[32][k]), k


def test_headline_pool_in_two_split_lanes(gpu_scene):
    """The benchmark's pool configuration: 776 candidates of 64 pieces x K = 32 through 776 slots, which the default
    lane threshold runs as two lanes of 388, both split. Bit-identical to the same batch through 128 slots in one
    fused lane. The batch's first four candidates are the ones test_headline_config_solve_against_the_oracle pins to
    the oracle (synthetic_batch seeds every candidate by its index)."""
    import topay_b200 as tp
    from topay_b200 import scenes
    n = 776
    opt = _headline_opt()
    paths, bv, ba = scenes.synthetic_batch(n, 1234)
    assert all(np.array_equal(a, b) for a, b in zip(paths, scenes.synthetic_batch(4, 1234)[0]))
    res, split = {}, {}
    for ns, lanes in ((n, 2), (128, 1)):
        s = tp.MomaTrajOpt(gpu_scene, max_cand=n, max_pieces=64, opt_param=opt, n_slots=ns)
        res[ns] = s.optimizeTrajBatch(paths, bv, ba)
        split[ns] = _split_batches(s.stats(), lanes)
        s.close()
    print(f"split lane-batches: {split}")
    assert split[n] >= 2 and split[128] == 0
    _assert_same_results(res[n], res[128], "776 slots in two lanes vs 128 slots")
    assert (res[n]["status"][:4] == 1).all()


def test_sweep_pool_in_two_split_lanes():
    """The sweep's configuration: eight scenarios with their own fields, 100 candidates each, in one upload through
    800 slots: two split lanes whose k_penalty is the MULTI variant (each candidate reads its own scenario's field).
    Every scenario's winner, trajectory and both gate verdicts, and the results of all its candidates, are
    bit-identical to solving that scenario alone."""
    import topay_b200 as tp
    from topay_b200 import scenes
    n_sc, n_c = 8, 100
    fields, plans, alone = [], [], []
    for sc in range(n_sc):
        g = tp.GridMap(tp.grid_desc())
        g.regenerateMap(scenes.tables_scene(90 + sc)[0] if sc % 2 == 0 else scenes.cuboids_scene(90 + sc)[0])
        fields.append(g)
        plans.append(scenes.short_candidates(n_c, 5000 + sc))
        one = tp.MomaTrajOpt(g, max_cand=n_c, max_pieces=16)
        alone.append((one.planWinners([plans[sc]], use_gate=True)[0], {k: v.copy() for k, v in one.constraints.items()},
                      one.download()))
        assert _split_batches(one.stats(), 1) == 0
        one.close()
    pool = tp.MomaTrajOpt(fields[0], max_cand=n_sc * n_c, max_pieces=16, n_slots=n_sc * n_c)
    got = pool.planWinners(plans, use_gate=True, fields=fields)
    split = _split_batches(pool.stats(), 2)
    print(f"split lane-batches: {split}")
    assert split >= 2
    gate, res = pool.constraints, pool.download()
    for sc in range(n_sc):
        w, (a, ag, ar) = got[sc], alone[sc]
        _assert_same_winner(a, w, sc)
        sl = slice(sc * n_c, (sc + 1) * n_c)
        for k in ("feasible", "feasible_print"):
            assert np.array_equal(gate[k][sl], ag[k]), (sc, k)
        _assert_same_results({k: res[k][sl] for k in RESULT_KEYS}, ar, sc)
    assert any(w is not None for w in got)
    pool.close()
    for g in fields:
        g.close()


def test_timed_mode_at_the_headline_size(gpu_scene):
    """The four headline candidates (64 pieces x K = 32), graph mode against timed mode (plain launches, k_cand always
    split, the L-BFGS launch with a ring sized by its own shared memory): bit-identical results and L-BFGS trace,
    and the timed run reports a time for each half of k_cand."""
    import topay_b200 as tp
    from topay_b200 import scenes
    n = 4
    paths, bv, ba = scenes.synthetic_batch(n, 1234)
    s = tp.MomaTrajOpt(gpu_scene, max_cand=n, max_pieces=64, opt_param=_headline_opt())
    s.set_trace(20000)
    graph = s.optimizeTrajBatch(paths, bv, ba)
    assert _split_batches(s.stats(), 1) == 0
    graph_trace = [s.trace(c) for c in range(n)]
    s.set_timed(True)
    timed = s.optimizeTrajBatch(paths, bv, ba)
    st = s.stats()
    assert st["kernel_launches"] == 2 + SPLIT * st["ticks"] // 16 and st["eval_launches"] == st["ticks"], st
    assert st["ms_adj"] > 0 and st["ms_lbfgs"] > 0 and st["ms_gen"] > 0, st
    _assert_same_results(graph, timed, "graph vs timed")
    for c in range(n):
        assert len(graph_trace[c]) > 15 and np.array_equal(s.trace(c), graph_trace[c]), c
    assert (timed["status"] == 1).all()
    s.close()
