"""First success + grace and stops in a streaming session, on one GPU: bench.latency_probe's 200 reference-scale plans
(8 candidates, same seeds as scripts/stream_probe.py) submitted one every 5 ms into one pool, with the gate.

- grace off and G = 0, 100, 500 (topay_solver_stream_set_grace): p50 / p90 latency submit -> poll, plans with a
  winner, and against grace off how many winners (index by duration) changed and the mean relative change of the
  winner's duration over the plans that have a winner both ways;
- grace off, every plan stopped 60 ms after its submission (topay_solver_stream_stop): the same figures.

Each setting runs a warm-up session first (its graphs captured). Prints one JSON object; --out also writes it to a file.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    sys.path.insert(0, p)

from grace_probe import card  # noqa: E402

CAND, N_PLANS, INTERVAL_MS, STOP_MS = 8, 200, 5.0, 60.0
GRACES = (None, 0, 100, 500)


def session(s, plans, grace, stop_ms=None, interval_ms=INTERVAL_MS):
    """One session: plan i submitted at i * interval_ms, each stopped stop_ms after its submission if given; every
    winner is taken as it is reported. Returns per plan (latency ms, winner index, winner duration)."""
    t_sub, out, ids, stopped, i = {}, {}, {}, set(), 0
    s.stream_begin(use_gate=True, grace_evals=grace)
    t0 = time.perf_counter()
    for _ in range(10000000):
        now = time.perf_counter()
        while i < len(plans) and now - t0 >= i * interval_ms * 1e-3:
            pid = s.stream_submit(*plans[i])
            ids[pid], t_sub[i] = i, time.perf_counter()
            i += 1
        if stop_ms is not None:
            now = time.perf_counter()
            for pid, p in ids.items():
                if pid not in stopped and (now - t_sub[p]) * 1e3 >= stop_ms:
                    s.stream_stop(pid)
                    stopped.add(pid)
        live = s.stream_advance(1)
        for pid, bd, _ in s.stream_poll():
            p = ids.pop(pid)
            stopped.discard(pid)
            r = s.stream_take(pid, cand=max(bd, 0))
            out[p] = ((time.perf_counter() - t_sub[p]) * 1e3, bd, float(r["duration"]) if bd >= 0 else float("nan"))
        if i == len(plans) and not ids and live == 0:
            break
        if live == 0 and i < len(plans):
            time.sleep(max(0.0, t0 + i * interval_ms * 1e-3 - time.perf_counter()))
    s.stream_end()
    return [out[p] for p in range(len(plans))]


def summary(runs, base):
    lat = np.array([r[0] for r in runs])
    out = {"p50_ms": float(np.median(lat)), "p90_ms": float(np.percentile(lat, 90)),
           "plans_with_a_winner": int(sum(r[1] >= 0 for r in runs))}
    if base is not None:
        rel = [(b[2] - a[2]) / a[2] for a, b in zip(base, runs) if a[1] >= 0 and b[1] >= 0]
        out.update({"winners_changed": int(sum(a[1] != b[1] for a, b in zip(base, runs))),
                    "plans_that_lost_their_winner": int(sum(a[1] >= 0 and b[1] < 0 for a, b in zip(base, runs))),
                    "mean_rel_duration_change": float(np.mean(rel)) if rel else None})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import topay_b200 as tp
    from topay_b200 import scenes
    gm = tp.GridMap(tp.grid_desc(), device=0)
    pts, _ = scenes.cuboids_scene(42)
    gm.regenerateMap(pts)
    plans = [scenes.short_candidates(CAND, 5000 + p) for p in range(5, N_PLANS + 5)]
    pool = tp.MomaTrajOpt(gm, max_cand=N_PLANS * CAND, max_pieces=16)
    out = {"card": card(), "plans": N_PLANS, "candidates": CAND, "interval_ms": INTERVAL_MS, "use_gate": True}
    base = None
    for g in GRACES:
        session(pool, plans[:20], g, interval_ms=0)      # warm-up: graphs of the launch grids
        runs = session(pool, plans, g)
        if g is None:
            base = runs
        out["off" if g is None else f"G={g}"] = summary(runs, None if g is None else base)
    session(pool, plans[:20], None, STOP_MS, interval_ms=0)
    out[f"off_stop_after_{int(STOP_MS)}ms"] = summary(session(pool, plans, None, STOP_MS), base)
    pool.close()
    gm.close()
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
