"""Streaming sessions (topay_solver_stream_*) against the batch paths they replace, on one GPU, in one process:

- sweep: bench.sweep_probe's 512 scenarios x 8 candidates. The grouped shared solve is bench.sweep_probe itself; the
  stream builds each scenario's field and submits its plan, advancing one batch between builds. Both alternate twice.
  The per-scenario winners (index by duration) must be identical between the two.
- arrivals: bench.latency_probe's 200 reference-scale plans, submitted back to back and one every 5 ms into one pool,
  latency = submit -> poll; next to bench.latency_probe (one run per plan).

Prints one JSON object; --out also writes it to a file. The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import bench  # noqa: E402
from grace_probe import card  # noqa: E402

N_SCEN, CAND, N_PLANS = 512, 8, 200


def sweep_inputs(scenes):
    """bench.sweep_probe's scenarios (one rank): clouds and candidates of the same seeds."""
    clouds = [scenes.tables_scene(s)[0] if s % 2 == 0 else scenes.cuboids_scene(s)[0] for s in range(N_SCEN)]
    cands = [scenes.short_candidates(CAND, 100000 + s) for s in range(N_SCEN)]
    return clouds, cands


def sweep_stream(tp, s, fields, clouds, cands):
    """Build a scenario's field, submit its plan, advance one batch; then drain. Returns (seconds, winners)."""
    import torch
    win, ids = [None] * N_SCEN, {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.stream_begin(use_gate=True)
    for i in range(N_SCEN):
        fields[i].regenerateMap(clouds[i])
        ids[s.stream_submit(*cands[i], field=fields[i])] = i
        s.stream_advance(1)
        for pid, bd, _ in s.stream_poll():
            win[ids.pop(pid)] = bd
            s.stream_take(pid, cand=max(bd, 0))       # the winner crosses the bus
    for _ in range(100000):
        live = s.stream_advance(1)
        for pid, bd, _ in s.stream_poll():
            win[ids.pop(pid)] = bd
            s.stream_take(pid, cand=max(bd, 0))
        if live == 0 and not ids:
            break
    s.stream_end()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, win


def arrivals(s, plans, interval_ms):
    """Submit every plan (back to back, or one every interval_ms while advancing); latency = submit -> poll."""
    t_sub, lat, ids, i = {}, {}, {}, 0
    s.stream_begin(use_gate=True)
    t0 = time.perf_counter()
    for _ in range(1000000):
        now = time.perf_counter()
        while i < len(plans) and (interval_ms == 0 or now - t0 >= i * interval_ms * 1e-3):
            pid = s.stream_submit(*plans[i])
            ids[pid], t_sub[i] = i, time.perf_counter()
            i += 1
        live = s.stream_advance(1)
        for pid, bd, _ in s.stream_poll():
            p = ids.pop(pid)
            s.stream_take(pid, cand=max(bd, 0))
            lat[p] = (time.perf_counter() - t_sub[p]) * 1e3
        if i == len(plans) and not ids and live == 0:
            break
        if live == 0 and i < len(plans):
            time.sleep(max(0.0, t0 + i * interval_ms * 1e-3 - time.perf_counter()))
    s.stream_end()
    v = np.array([lat[p] for p in range(len(plans))])
    return {"p50_ms": float(np.median(v)), "p90_ms": float(np.percentile(v, 90)),
            "seconds": time.perf_counter() - t0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import topay_b200 as tp
    from topay_b200 import scenes
    out = {"card": card()}
    clouds, cands = sweep_inputs(scenes)
    fields = []
    for _ in range(N_SCEN):
        g = tp.GridMap(tp.grid_desc(), device=0)
        g.set_keep_sqdist(False)
        fields.append(g)
    s = tp.MomaTrajOpt(fields[0], max_cand=N_SCEN * CAND, max_pieces=16)
    # the grouped solve's winners on the same scenarios, for the identity check
    for f, c in zip(fields, clouds):
        f.regenerateMap(c)
    grouped_win = [w["index"] if w is not None else -1 for w in s.planWinners(cands, use_gate=True, fields=fields)]
    rounds = []
    for r in range(2):
        g = bench.sweep_probe(tp, scenes, 0, 0, 1, None)
        dt, win = sweep_stream(tp, s, fields, clouds, cands)
        assert win == grouped_win, "stream winners differ from the grouped solve's"
        rounds.append({"grouped_scenarios_per_s": g["scenarios_per_s"], "stream_scenarios_per_s": N_SCEN / dt})
    s.close()
    for f in fields:
        f.close()
    out["sweep"] = {"scenarios": N_SCEN, "candidates": CAND, "rounds": rounds, "winners_identical": True,
                    "scenarios_with_a_feasible_winner": int(sum(w >= 0 for w in grouped_win))}
    gm = tp.GridMap(tp.grid_desc(), device=0)
    pts, _ = scenes.cuboids_scene(42)
    gm.regenerateMap(pts)
    plans = [scenes.short_candidates(CAND, 5000 + p) for p in range(5, N_PLANS + 5)]
    pool = tp.MomaTrajOpt(gm, max_cand=N_PLANS * CAND, max_pieces=16)
    arrivals(pool, plans[:20], 0)                       # warm-up: graphs of the launch grids
    out["arrivals"] = {"one_run_per_plan": bench.latency_probe(tp, scenes, gm),
                       "stream_back_to_back": arrivals(pool, plans, 0),
                       "stream_every_5ms": arrivals(pool, plans, 5)}
    pool.close()
    gm.close()
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
