"""A replanning loop on the reference-size ROG-Map ring (803 x 803 x 83 at 0.05 m), on one GPU: a ProbMap ingests one
cuboids-scene cloud of 10^5 points every 100 ms (updateProbMap, which rebuilds the ring), and a reference-scale plan
(8 candidates, bench.latency_probe's kind) is due every 50 ms into one streaming session of a ROG solver with the gate.

- snapshots (topay_solver_stream_set_snapshots): frames are applied when due and plans submitted when due, each pinned
  to the ring of its submit;
- hold: the schedule that is safe without snapshots. A due frame waits until every submitted plan has been taken, and
  no plan is submitted while a frame waits.

Reported per schedule: due -> poll latency p50 / p90 of the plans (from the time the plan was due, so a held submit
counts), map staleness (due -> applied time of the frames, and how many frames were waiting when one was applied),
submits refused because every snapshot was held. Also the device time of one snapshot copy (the three device-to-device
copies of dist3, crit and flat, from a torch.profiler trace of a separate short run). Prints one JSON object; --out also
writes it to a file. The card's name and power limit are read in the same run."""
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
from topay_b200._lib import ERR_TOO_LARGE, TopayError  # noqa: E402

CAND, FRAME_MS, PLAN_MS, POINTS = 8, 100.0, 50.0, 100000


def world(tp, scenes, n_frames, seed=3):
    """The ring, its ProbMap, and the frames: (cloud, pose) with the robot moving 2 cm per frame."""
    esdf = tp.ESDFMap(tp.rog_desc(map_sliding_en=True))
    prob = tp.ProbMap(esdf, tp.prob_desc(ray_range=(0.3, 10.0), inflation_resolution=0.05))
    rng = np.random.default_rng(seed)
    frames, scene = [], [scenes.cuboids_scene(seed + k)[0] for k in range(4)]
    for k in range(n_frames):
        pts = scene[k % 4]
        pts = pts[rng.choice(len(pts), min(POINTS, len(pts)), replace=False)].astype(np.float64) - [10.0, 10.0, 0.0]
        pose = np.array([0.02 * k, 0.0, 0.4])
        frames.append((np.concatenate([pts, rng.uniform(0, 100, (len(pts), 1))], axis=1).astype(np.float32), pose))
    return esdf, prob, frames


def run(tp, s, prob, frames, plans, mode, seconds):
    """One session of `seconds`; returns the latencies of the plans and the staleness of the frames."""
    s.stream_begin(use_gate=True, snapshots=6 if mode == "snapshots" else 0)
    due_plan, lat, ids, fi, pi, refused = {}, [], {}, 0, 0, 0
    waiting, stale_ms, held = [], [], []
    t0 = time.perf_counter()
    while True:
        now = (time.perf_counter() - t0) * 1e3
        if now > seconds * 1e3 and not ids:
            break
        while fi < len(frames) and now >= fi * FRAME_MS and now <= seconds * 1e3:
            waiting.append((fi, fi * FRAME_MS))
            fi += 1
        if waiting and (mode == "snapshots" or not ids):
            for k, due in waiting:
                held.append(len(waiting))
                prob.updateProbMap(*frames[k])
                stale_ms.append((time.perf_counter() - t0) * 1e3 - due)
            waiting = []
        if now <= seconds * 1e3 and now >= pi * PLAN_MS and (mode == "snapshots" or not waiting):
            try:
                pid = s.stream_submit(*plans[pi % len(plans)])
                ids[pid], due_plan[pid] = pi, pi * PLAN_MS
                pi += 1
            except TopayError as e:
                if e.code != ERR_TOO_LARGE:
                    raise
                refused += 1
        s.stream_advance(1)
        for pid, _, _ in s.stream_poll():
            lat.append((time.perf_counter() - t0) * 1e3 - due_plan.pop(pid))
            s.stream_take(pid, gate=True)
            ids.pop(pid)
    s.stream_end()
    q = lambda a, p: round(float(np.percentile(a, p)), 2) if len(a) else None  # noqa: E731
    return {"plans": len(lat), "latency_ms_p50": q(lat, 50), "latency_ms_p90": q(lat, 90),
            "frames": len(stale_ms), "staleness_ms_p50": q(stale_ms, 50), "staleness_ms_p90": q(stale_ms, 90),
            "staleness_ms_max": q(stale_ms, 100), "frames_waiting_mean": round(float(np.mean(held)), 2) if held else None,
            "frames_waiting_max": int(max(held)) if held else None, "submits_refused": refused}


def copy_time(tp, s, prob, frames, plans, n=8):
    """Device time of the snapshot copies of n submits, each after a frame: torch.profiler's CUDA activity of the
    device-to-device copies (every stream of the process is traced)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    s.stream_begin(use_gate=True, snapshots=2)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for k in range(n):
            prob.updateProbMap(*frames[k])
            pid = s.stream_submit(*plans[k])
            for _ in range(100000):
                s.stream_advance(4)
                if s.stream_poll():
                    break
            s.stream_take(pid)
        torch.cuda.synchronize()
    s.stream_end()
    us = [e.time_range.elapsed_us() for e in prof.events() if "Memcpy DtoD" in e.name]
    us = sorted(us, reverse=True)
    if not us:
        return {"snapshot_copy_ms": None, "note": "no device-to-device copy in the trace"}
    big = us[:n]
    return {"snapshot_copy_ms": round(sum(us[:3 * n]) / n / 1e3, 4), "dist3_copy_ms": round(float(np.mean(big)) / 1e3, 4),
            "copies_traced": len(us), "bytes_per_snapshot": 803 * 803 * 83 * 8 + 2 * 803 * 803 * 8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=8.0)
    ap.add_argument("--out")
    args = ap.parse_args()
    import topay_b200 as tp
    from topay_b200 import scenes
    n_frames = int(args.seconds * 1e3 / FRAME_MS) + 2
    esdf, prob, frames = world(tp, scenes, n_frames)
    prob.updateProbMap(*frames[0])
    plans = [scenes.short_candidates(CAND, 7100 + p) for p in range(40)]
    s = tp.MomaTrajOpt(esdf, max_cand=64 * CAND, max_pieces=16)
    out = {"card": card(), "ring": list(esdf.map_size_i), "frame_ms": FRAME_MS, "plan_ms": PLAN_MS,
           "points_per_frame": int(len(frames[0][0]))}
    run(tp, s, prob, frames, plans, "snapshots", 1.0)          # warm-up: graphs captured, pools grown
    out["copy"] = copy_time(tp, s, prob, frames, plans)
    for mode in ("snapshots", "hold", "snapshots", "hold"):     # alternated twice
        out.setdefault(mode, []).append(run(tp, s, prob, frames, plans, mode, args.seconds))
    s.close()
    prob.close()
    esdf.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
