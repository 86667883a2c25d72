"""First success + grace (topay_solver_set_plans): latency, throughput and winner quality with grace off and at
G = 0, 100, 500 evaluations, on one GPU.

- latency: bench.latency_probe's 200 reference-scale plans (8 candidates, same seeds) through optimizeTrajBatch;
- the lone 256-candidate headline plan (64 pieces x K = 32): ticks and wall time;
- headline-pool throughput: 8 plans of 256 through 2048 slots;
- for each G, how many per-plan winners (shortest duration among status-1 candidates) changed against grace off, and
  the mean relative change of the winner's duration over the plans that have a winner both ways;
- the oracle port's CPU time per evaluation at reference scale (one core), to read the reference's 100 ms grace in
  evaluations.

Prints one JSON object; --out also writes it to a file. The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

GRACES = (None, 0, 100, 500)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return {"name": "unknown", "power_limit": "unknown"}


def winners(res, off):
    """Per plan: (index of the shortest status-1 candidate, its duration), or (-1, nan)."""
    out = []
    for p in range(len(off) - 1):
        st, dur = res["status"][off[p]:off[p + 1]], res["duration"][off[p]:off[p + 1]]
        ok = np.flatnonzero(st == 1)
        out.append((int(ok[np.argmin(dur[ok])]), float(dur[ok].min())) if len(ok) else (-1, float("nan")))
    return out


def quality(base, got):
    changed = sum(a[0] != b[0] for a, b in zip(base, got))
    lost = sum(a[0] >= 0 and b[0] < 0 for a, b in zip(base, got))
    rel = [(b[1] - a[1]) / a[1] for a, b in zip(base, got) if a[0] >= 0 and b[0] >= 0]
    return {"winners_changed": changed, "plans_that_lost_their_winner": lost,
            "mean_rel_duration_change": float(np.mean(rel)) if rel else None}


def headline_opt(tp):
    opt = tp.opt_params_default()
    opt.int_K, opt.min_piece_num, opt.sample_interval = 32, 64, 1e9
    return opt


def latency(tp, scenes, gm, n_plans):
    s = tp.MomaTrajOpt(gm, max_cand=8, max_pieces=16)
    out, base = {}, None
    for g in GRACES:
        lat, win = [], []
        for plan in range(n_plans + 5):
            paths, bv, ba = scenes.short_candidates(8, 5000 + plan)
            t0 = time.perf_counter()
            r = s.optimizeTrajBatch(paths, bv, ba, grace_evals=g)
            dt = (time.perf_counter() - t0) * 1e3
            if plan >= 5:
                lat.append(dt)
                win += winners(r, [0, 8])
        key = "off" if g is None else f"G={g}"
        out[key] = {"p50_ms": float(np.median(lat)), "p90_ms": float(np.percentile(lat, 90)),
                    "plans_with_a_winner": sum(w[0] >= 0 for w in win)}
        if g is None:
            base = win
        out[key].update(quality(base, win))
    s.close()
    return out


def lone_plan(tp, scenes, gm):
    paths, bv, ba = scenes.synthetic_batch(256, 1234)
    s = tp.MomaTrajOpt(gm, max_cand=256, max_pieces=64, opt_param=headline_opt(tp))
    out, base = {}, None
    for g in GRACES:
        s.upload(paths, bv, ba)
        s.set_plans(None, g)
        s.run()
        t0 = time.perf_counter()
        s.run()
        dt = time.perf_counter() - t0
        r = s.download()
        key = "off" if g is None else f"G={g}"
        w = winners(r, [0, 256])
        out[key] = {"ms": dt * 1e3, "ticks": int(s.stats()["ticks"]), "successes": int((r["status"] == 1).sum())}
        if g is None:
            base = w
        out[key].update(quality(base, w))
    s.close()
    return out


def pool(tp, scenes, gm):
    plans = [scenes.synthetic_batch(256, 1234 + 1000 * p) for p in range(8)]
    paths = [q for p in plans for q in p[0]]
    bv, ba = np.concatenate([p[1] for p in plans]), np.concatenate([p[2] for p in plans])
    off = np.arange(0, 2049, 256, dtype=np.int32)
    s = tp.MomaTrajOpt(gm, max_cand=2048, max_pieces=64, opt_param=headline_opt(tp), n_slots=2048)
    s.upload(paths, bv, ba)
    s.run()                 # warm-up: graphs instantiated
    out, base = {}, None
    for g in GRACES:
        s.upload(paths, bv, ba)
        s.set_plans(off, g)
        t0 = time.perf_counter()
        s.run()
        dt = time.perf_counter() - t0
        r = s.download()
        key = "off" if g is None else f"G={g}"
        w = winners(r, off)
        out[key] = {"trajectories_per_s": 2048 / dt, "ms": dt * 1e3, "ticks": int(s.stats()["ticks"])}
        if g is None:
            base = w
        out[key].update(quality(base, w))
    s.close()
    return out


def oracle_eval_ms(tp, scenes, pts):
    """CPU time of one stage-2 cost/gradient evaluation of the oracle port at reference scale."""
    import oracle_lib as O
    desc = tp.grid_desc()
    of = O.Field(desc)
    of.rasterize(pts)
    of.rebuild()
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    paths, bv, ba = scenes.short_candidates(8, 5000)
    prep = [tp.prepare_candidate(opt, rp, p, bv[0], ba[0], 16) for p in paths]
    reps = 50
    t0 = time.process_time()
    for _ in range(reps):
        for q in prep:
            N = q["piece_num"]
            O.eval_one(opt, rp, of, 2, N, q["head_pva"], q["tail_pva"], q["start_xy"], q["end_xy"],
                       q["init_inner_xy"][:N], np.zeros(2), np.full(2, 1e4), q["x0"])
    ms = (time.process_time() - t0) * 1e3 / (reps * len(prep))
    return {"ms_per_eval": ms, "evals_in_100ms": 100.0 / ms,
            "pieces": [int(q["piece_num"]) for q in prep], "note": "one core, process CPU time, stage 2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--plans", type=int, default=200)
    ap.add_argument("--out")
    args = ap.parse_args()
    import topay_b200 as tp
    from topay_b200 import scenes
    pts, _ = scenes.cuboids_scene(42)
    gm = tp.GridMap(tp.grid_desc())
    gm.regenerateMap(pts)
    line = {"card": card(), "graces": ["off" if g is None else g for g in GRACES],
            "latency_reference_scale": latency(tp, scenes, gm, args.plans),
            "lone_headline_plan": lone_plan(tp, scenes, gm),
            "headline_pool_8x256_2048_slots": pool(tp, scenes, gm),
            "oracle_cpu": oracle_eval_ms(tp, scenes, pts)}
    gm.close()
    print(json.dumps(line, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
