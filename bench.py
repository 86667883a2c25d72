#!/usr/bin/env python
"""Benchmark of the hot path: batched NLP solve of topological path candidates.

Workload (BASELINE.json configs[2], the one the metric "optimized trajectories/sec at 256
candidates" is quoted on): 256 synthetic S-curve candidates per GPU through a seeded cuboids scene
(20 x 20 x 1.6 m field @ 0.1 m), 64 pieces x int_K = 32 each (n = 632 variables), fp64, stage 1 +
stage-2 ALM to a terminal L-BFGS status. One "step" = one batched solve of all 256 candidates.

  python bench.py [--gpus N] [--steps K] [--warmup W]           device arm (this repo)
  python bench.py --impl reference [...]                        the reference's CPU algorithm
                                                                (oracle port) on the host cores

N > 1 is launched by torch.distributed.run, one rank per GPU; candidates shard across ranks with
no data-path collective (weak scaling: 256 per GPU), only timing is reduced (max over ranks).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_CAND, N_PIECES, INT_K = 256, 64, 32
NODE_BYTES = 800          # algorithmic ESDF bytes per penalty node, SURVEY.md §8(d)
NODE_FLOP = 4.0e3         # algorithmic fp64 flop per penalty node, SURVEY.md §8(d)
MID_FLOP = 0.15e3         # ... per Simpson midpoint node


def workload_params(tp):
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    opt.int_K = INT_K
    opt.min_piece_num = N_PIECES       # sample_interval chosen so that piece_num = 64 (SURVEY §8d)
    opt.sample_interval = 1e9
    return opt, rp


def base_config(n_cand):
    """The `config` object both arms print (the device arm's scheduling details go under `details`)."""
    return {"workload": f"synthetic {n_cand}-candidate batch per GPU, {N_PIECES} pieces x int_K {INT_K}, cuboids scene "
                        f"200x200x16 @0.1 m (BASELINE configs[2])",
            "candidates_per_gpu": n_cand, "pieces": N_PIECES, "int_K": INT_K, "variables": 10 * N_PIECES - 8}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    return rank, world, local, dist


def barrier_max(dist, local, value):
    """barrier + max over ranks of a python float (identity at world size 1)."""
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


class CpuArm:
    """The reference's CPU solve of the path on the host cores, thread per candidate like planner.cpp:921-925.
    kind "port" (default): the oracle's C++ restatement, bit-identical to the reference's own code
    (tests/test_ref_pin.py). kind "reference" (TOPAY_BENCH_CPU_REF=1): oracle/_ref/libtopay_ref.so — the reference's
    moma_traj_opt.cpp / grid_map.cpp compiled unmodified. That build links against this repo's Eigen STAND-IN
    (oracle/ref_stubs: plain loops over heap matrices, no expression templates), so its speed is the stand-in's, not
    Eigen's: measured 0.114 trajectories/s on 16 cores against 1.5 for the port. Timing it would inflate the GPU/CPU
    ratio 13-fold, so the timed CPU arm is the port and the compiled reference stays what it is for: the bit-level
    pin of the oracle. Checker / baseline code only."""

    def __init__(self, desc, pts):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        self.O = O
        self.rp = O.robot_defaults()
        self.of = O.Field(desc)
        self.of.rasterize(pts)
        self.of.rebuild()
        self.kind, self.R, self.grid = "port", None, None
        if os.environ.get("TOPAY_BENCH_CPU_REF") == "1" and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libtopay_ref.so")):
            try:
                import ref_lib as R
                self.grid = R.GridMap(desc)
                self.grid.set_cloud(pts)
                self.R, self.kind = R, "reference"
            except Exception as e:   # noqa: BLE001 — fall back to the port, say why
                print(f"bench: oracle/_ref unusable ({e}); CPU arm = oracle port", file=sys.stderr)

    def solve_batch(self, opt, paths, bv, ba, n_threads, wall_clock=False):
        """-> list of dicts with at least status. wall_clock: the reference's own 1.0 s ALM cap
        (moma_traj_opt.cpp:403) on the real clock instead of the deterministic alm_max_rounds."""
        if self.R is not None:
            return self.R.solve_batch(self.grid, opt, paths, bv, ba, n_threads, alm_max_rounds=opt.alm_max_rounds,
                                      wall_clock=wall_clock)
        return self.O.solve_batch(opt, self.rp, self.of, paths, bv, ba, n_threads=n_threads,
                                  wall_cap_s=1.0 if wall_clock else 0.0)

    def gate_pass(self, opt, paths, bv, ba, max_pieces):
        """Both verdicts of the worker's success gate (planner.cpp:877-880) on the CPU solves of these candidates
        (oracle solve = the reference's, bit for bit; its trajectories are what the gate needs)."""
        import threading
        res = [None] * len(paths)

        def work(c):
            res[c] = self.O.solve_one(opt, self.rp, self.of, paths[c], bv[c], ba[c], max_pieces=max_pieces)

        th = [threading.Thread(target=work, args=(c,)) for c in range(len(paths))]
        [t.start() for t in th]
        [t.join() for t in th]
        g = self.O.check_feasible(self.of, self.rp, [(r["T"], r["coeff"], paths[c][0, :3]) for c, r in enumerate(res)])
        ok = np.array([r["status"] == 1 for r in res])
        return int((ok & (g["feasible_print"] != 0)).sum()), int(ok.sum())


def cpu_baseline(opt, rp, pts, paths, bv, ba, cores, desc):
    """The reference's CPU solve on a bounded sample: one candidate per host core."""
    arm = CpuArm(desc, pts)
    O = arm.O
    m = min(cores, len(paths))
    t0 = time.perf_counter()
    res = arm.solve_batch(opt, paths[:m], bv[:m], ba[:m], cores)
    dt = time.perf_counter() - t0
    # the launch-file-equivalent figure: the same sample with the reference's 1.0 s wall-clock ALM cap
    t0 = time.perf_counter()
    res_cap = arm.solve_batch(opt, paths[:m], bv[:m], ba[:m], cores, wall_clock=True)
    dt_cap = time.perf_counter() - t0
    # success gate of the CPU solves of the first candidates (what the device's pass count is compared with)
    n_gate = min(m, 8)
    gate_ok, solved = arm.gate_pass(opt, paths[:n_gate], bv[:n_gate], ba[:n_gate], N_PIECES)
    # single-plan latency of the same algorithm at the reference's default scale (8 candidates on 8 threads,
    # planner.cpp:921-925), same plans as latency_probe
    from topay_b200 import scenes
    o2, lat = O.opt_defaults(), []
    for plan in range(8):
        p8, bv8, ba8 = scenes.short_candidates(8, 5005 + plan)
        t1 = time.perf_counter()
        arm.solve_batch(o2, p8, bv8, ba8, min(8, cores))
        lat.append((time.perf_counter() - t1) * 1e3)
    return {"value": m / dt, "unit": "trajectories/s", "cores": cores, "kind": arm.kind,
            "sample": f"{m} of the {len(paths)} candidates, one per host core (thread per candidate), {dt:.1f} s, "
                      f"{sum(r['status'] for r in res)} succeeded",
            "with_1s_alm_cap": {"value": m / dt_cap, "seconds": dt_cap, "succeeded": int(sum(r["status"] for r in res_cap)),
                                "note": "same sample under the reference's own 1.0 s wall-clock ALM cap "
                                        "(moma_traj_opt.cpp:403) instead of the deterministic alm_max_rounds"},
            "success_gate": {"candidates": n_gate, "solved": solved, "passed": gate_ok,
                             "note": "optimizeTraj && printConstraintsSituations (planner.cpp:877-880) on the CPU "
                                     "solves of the first candidates of the plan"},
            "latency_p50_ms": float(np.median(lat)),
            "latency_sample": "8 plans of 8 candidates on 8 threads, reference scale"}


def latency_probe(tp, scenes, gm, n_plans=200):
    """Second headline metric: p50 single-plan latency, upload candidates -> best trajectory on the
    host, at the reference's default scale (BASELINE configs[0]/[1]: <= 8 candidates per plan,
    int_K = 12, sample_interval 1.5 s -> 3-10 pieces), one plan at a time through the public API."""
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    solver = tp.MomaTrajOpt(gm, max_cand=8, max_pieces=16, opt_param=opt, robot=rp)
    lat, ok = [], 0
    for plan in range(n_plans + 5):
        paths, bv, ba = scenes.short_candidates(8, 5000 + plan)
        t0 = time.perf_counter()
        r = solver.optimizeTrajBatch(paths, bv, ba)
        dt = (time.perf_counter() - t0) * 1e3
        if plan >= 5:
            lat.append(dt)
            ok += int(r["best_by_duration"] >= 0)
    lat = np.array(lat)
    solver.close()
    return {"p50_ms": float(np.median(lat)), "p90_ms": float(np.percentile(lat, 90)), "plans": n_plans,
            "plans_with_a_feasible_winner": ok,
            "workload": "8 candidates per plan, int_K 12, 3-10 pieces, cuboids scene 200x200x16 (reference scale)"}


def field_probe(tp, scenes, device, hbm_peak):
    """BASELINE configs[3]: ESDF rebuild + query on the 40 x 40 x 4 m grid at 0.05 m (800 x 800 x 80)."""
    import torch
    desc = tp.grid_desc(map_size=(40.0, 40.0, 4.0), resolution=0.05)
    gm = tp.GridMap(desc, device=device)
    pts, _ = scenes.cuboids_scene(7, size_x=40.0, size_y=40.0, scale=2.0)
    gm.regenerateMap(pts)
    gm.set_keep_sqdist(False)
    t3 = []
    for _ in range(5):
        gm.updateESDF()
        t3.append(gm.last_rebuild_ms())
    tot, d3 = np.median([a for a, _ in t3]), np.median([b for _, b in t3])
    vox = 800 * 800 * 80
    # resident queries: 10^7 uniformly random in-map points (seed 7), value + gradient
    n = 10_000_000
    g = torch.Generator(device=f"cuda:{device}").manual_seed(7)
    lo = torch.tensor([-20.0, -20.0, 0.0], device=f"cuda:{device}", dtype=torch.float64)
    hi = torch.tensor([20.0, 20.0, 4.0], device=f"cuda:{device}", dtype=torch.float64)
    pos = lo + (hi - lo) * torch.rand((n, 3), generator=g, device=f"cuda:{device}", dtype=torch.float64)
    dist = torch.empty(n, device=f"cuda:{device}", dtype=torch.float64)
    grad = torch.empty((n, 3), device=f"cuda:{device}", dtype=torch.float64)
    import ctypes as C
    from topay_b200 import _lib
    l = _lib.lib()
    qms = []
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _lib.check(l.topay_field_query3d_dev(gm.h, C.c_void_p(pos.data_ptr()), n, C.c_void_p(dist.data_ptr()),
                                             C.c_void_p(grad.data_ptr())), "query3d_dev")
        _lib.check(l.topay_field_sync(gm.h), "sync")
        qms.append((time.perf_counter() - t0) * 1e3)
    q = float(np.median(qms[1:]))
    # the gather-bound regime of the solve: one 256-candidate plan of the headline workload evaluated against THIS
    # 410 MB field (12 trilinear lookups per penalty node no longer hit a 5 MB L2-resident grid), per-kernel times
    # from CUDA events around every launch
    opt, rp = workload_params(tp)
    paths, bv, ba = scenes.synthetic_batch(256, 1234)
    solver = tp.MomaTrajOpt(gm, max_cand=256, max_pieces=N_PIECES, opt_param=opt, robot=rp)
    solver.upload(paths, bv, ba)
    solver.set_timed(True)
    solver.run()
    st = solver.stats()
    big = {"workload": "one 256-candidate plan (64 pieces x int_K 32) solved against the 800x800x80 field, timed launches",
           "k_penalty_ns_per_node": 1e6 * st["ms_eval"] / max(st["eval_nodes"], 1),
           "k_penalty_algorithmic_GBps": st["eval_nodes"] * NODE_BYTES / max(st["ms_eval"] * 1e-3, 1e-12) / 1e9,
           "k_penalty_share": st["ms_eval"] / max(st["ms_eval"] + st["ms_lbfgs"] + st["ms_gen"] + st["ms_adj"] +
                                                  st["ms_chain"] + st["ms_integrate"], 1e-9),
           "successes": int(solver.download()["status"].sum())}
    solver.close()
    gm.close()
    return {"grid": "800x800x80 @0.05 m", "rebuild_ms_total": float(tot), "rebuild_ms_3d": float(d3), "solve_on_this_field": big,
            "rebuild_algorithmic_GBps": vox * 9 / (d3 * 1e-3) / 1e9, "rebuild_frac_of_hbm_peak": vox * 9 / (d3 * 1e-3) / 1e9 / hbm_peak,
            "query_ms_1e7": q, "query_Gpoints_per_s": n / (q * 1e-3) / 1e9,
            "query_algorithmic_GBps": n * (24 + 64 + 32) / (q * 1e-3) / 1e9,
            "note": "rebuild: 9 B/voxel algorithmic (1 B occupancy in, 8 B ESDF out); query: 24 B position + "
                    "8 taps x 8 B + 32 B result per point, points resident in HBM"}


def sweep_probe(tp, scenes, local, rank, world, dist, per_rank=512, candidates=8, group=512, workers=1):
    """BASELINE configs[4] (the scenario sweep, bounded): `per_rank` x world independent table / cuboid scenarios,
    static round-robin over the ranks (one process per GPU, no data-path collective). Every scenario runs the whole
    device pipeline the planner drives: rasterise its point cloud -> rebuild ITS field (4 x 2-D + 3-D ESDF) -> solve
    its candidates -> success gate -> shortest feasible trajectory (selected on the device, the winner alone crosses
    the bus). Scenarios are taken `group` at a time: their fields are rebuilt one after the other, then the candidates
    of the whole group share ONE device solve, each read against its own scenario's field
    (topay_solver_assign_fields) — the launches of a tick are paid once per group instead of once per scenario.
    `workers` groups are in flight. Measured on one B200 (512 scenarios): one scenario per solve, 32 solves in flight 94
    scenarios/s; 64 per solve 210; 128: 263; 512: 295 (field builds 0.57 ms per scenario, the shared solve is bound by
    its slowest candidate: 2350 ticks of 340 us). The per-scenario winners (scenario,
    index, duration, cost: 32 B each) are then gathered on every rank, over NCCL and over the host (gloo), both timed:
    north_star uses NCCL only if it measurably wins."""
    import threading
    import torch
    from topay_b200 import shard
    total = per_rank * world
    mine = shard.round_robin(total, rank, world)
    group = max(1, min(group, len(mine)))
    groups = [mine[i:i + group] for i in range(0, len(mine), group)]
    P = max(1, min(workers, len(groups)))
    opt, rp = tp.opt_params_default(), tp.robot_params_default()
    slots = []
    for _ in range(P):
        fields = []
        for _ in range(group):
            g = tp.GridMap(tp.grid_desc(), device=local)
            g.set_keep_sqdist(False)
            fields.append(g)
        slots.append((fields, tp.MomaTrajOpt(fields[0], max_cand=group * candidates, max_pieces=16, opt_param=opt, robot=rp)))
    clouds = {s: (scenes.tables_scene(s)[0] if s % 2 == 0 else scenes.cuboids_scene(s)[0]) for s in mine}
    cands = {s: scenes.short_candidates(candidates, 100000 + s) for s in mine}
    out, lock = {}, threading.Lock()

    def worker(slot):
        fields, solver = slots[slot]
        for grp in groups[slot::P]:
            for f, s in zip(fields, grp):
                f.regenerateMap(clouds[s])
            ws = solver.planWinners([cands[s] for s in grp], use_gate=True, fields=fields[:len(grp)])
            with lock:
                for s, w in zip(grp, ws):
                    out[s] = (float(w["index"]), float(w["duration"]), float(w["cost"])) if w is not None else (-1.0, 0.0, 0.0)

    for warm in (True, False):        # one untimed pass (graphs, allocations), one timed
        out.clear()
        barrier_max(dist, local, 0.0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        th = [threading.Thread(target=worker, args=(i,)) for i in range(P)]
        [t.start() for t in th]
        [t.join() for t in th]
        torch.cuda.synchronize()
        dt = barrier_max(dist, local, time.perf_counter() - t0)
    rows = torch.tensor([[float(s), *out[s]] for s in mine], dtype=torch.float64)
    gather = {"bytes_per_rank": int(rows.numel() * 8)}
    n_win = int((rows[:, 1] >= 0).sum())
    if dist is not None:
        dev_rows = rows.to(f"cuda:{local}")
        gl = dist.new_group(backend="gloo")
        for name, t_in, grp in (("nccl", dev_rows, None), ("host_gloo", rows, gl)):
            bufs = [torch.empty_like(t_in) for _ in range(world)]
            ts = []
            for _ in range(30):
                if name == "nccl":
                    torch.cuda.synchronize()
                t0 = time.perf_counter()
                dist.all_gather(bufs, t_in, group=grp)
                if name == "nccl":
                    torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e6)
            gather[name + "_us_p50"] = barrier_max(dist, local, float(np.median(ts[5:])))
            allr = torch.cat([b.cpu() for b in bufs])
        n_win = int((allr[:, 1] >= 0).sum())
        gather["faster"] = "nccl" if gather["nccl_us_p50"] < gather["host_gloo_us_p50"] else "host"
    for fields, solver in slots:
        solver.close()
        for g in fields:
            g.close()
    return {"workload": "scenario sweep (BASELINE configs[4], bounded): rasterise + field rebuild per scenario, the "
                        "candidates of a group of scenarios in one device solve (each against its own field) + "
                        "success gate + device-side selection per scenario, round-robin over ranks",
            "scenarios": total, "scenarios_per_gpu": per_rank, "candidates_per_scenario": candidates, "n_gpus": world,
            "scenarios_per_solve": group, "groups_in_flight_per_gpu": P, "scenarios_per_s": total / dt, "trajectories_per_s": total * candidates / dt,
            "scenarios_with_a_feasible_winner": n_win, "seconds": dt, "winner_gather": gather}


def subpath_probe(tp, scenes, device, hbm_peak, solver, gm, rp, with_cpu):
    """The other rows of SURVEY.md §8 next to the solve, each with the oracle timed beside it on a bounded
    sample (single host thread — these reference routines are serial): ROG-Map ring update (a23), field
    rebuild at the default grid (a20/a21), 3-D queries (a18), success gate (a16 + N1)."""
    from topay_b200.rog import ESDFMap
    out = {}
    rng = np.random.default_rng(0)
    # ---- ROG ring, 803 x 803 x 83 (SURVEY §8 a23)
    rog = ESDFMap(tp.rog_desc(), device=device)
    res = rog.resolution
    cells = np.stack(np.meshgrid(np.arange(0, 1, res), np.arange(0, 1, res), np.arange(0, 1.5, res), indexing="ij"), -1)
    pts = np.concatenate([rng.uniform([-18, -18, 0], [18, 18, 0.2]) + cells.reshape(-1, 3) for _ in range(60)])
    rog.updateGridCounter(pts, 1, 3)
    ms = []
    for odom in [(0, 0, 0), (0, 0, 0), (0.5, 0.3, 0.0), (0.5, 0.3, 0.0), (0.5, 0.3, 0.0)]:
        rog.mapSliding(odom)
        rog.updateESDF3D(odom)
        ms.append(rog.last_update_ms())
    tot, d3 = float(np.median([a for a, _ in ms[1:]])), float(np.median([b for _, b in ms[1:]]))
    vox = 800 * 800 * 80          # the update box (the ring is 803 x 803 x 83)
    out["rog_update"] = {"ring": "803x803x83 @0.05 m, update box 800x800x80, ring wrap on x and y",
                         "ms_total": tot, "ms_3d": d3, "Mvoxel_per_s": vox / (tot * 1e-3) / 1e6,
                         "algorithmic_GBps": vox * 9 / (d3 * 1e-3) / 1e9,
                         "frac_of_hbm_peak": vox * 9 / (d3 * 1e-3) / 1e9 / hbm_peak}
    # ---- ProbMap ingest (N3): lidar-like frames of 10^5 points into the probability ring that feeds the same ESDF ring
    from topay_b200.rog import ProbMap
    pm = ProbMap(rog, tp.prob_desc(ray_range=(0.3, 10.0), virtual_ceil_height=3.0, virtual_ground_height=-0.5,
                                   local_update_box=(20.0, 20.0, 4.0), inflation_resolution=res))
    dirs = rng.normal(size=(100000, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    cloud = np.concatenate([dirs * rng.uniform(0.5, 9.0, (100000, 1)) + np.array([0.0, 0.0, 1.0]),
                            np.full((100000, 1), 50.0)], axis=1).astype(np.float32)
    tms = []
    for k in range(4):
        t0 = time.perf_counter()
        pm.updateProbMap(cloud, (0.02 * k, 0.0, 1.0))
        tms.append((time.perf_counter() - t0) * 1e3)
    out["prob_map_update"] = {"frame": "10^5 points, rays up to 9 m at 0.05 m, ring 801x801x81 (incl. updateESDF3D of the "
                                       "update box)", "ms_per_frame": float(np.median(tms[1:])),
                              "Mpoints_per_s": 0.1 / (float(np.median(tms[1:])) * 1e-3)}
    pm.close()
    rog.close()
    # ---- success gate on the candidates of the last solve, resident
    t = []
    for _ in range(4):
        t0 = time.perf_counter()
        arrs, best = solver.checkFeasibleBatch()
        t.append((time.perf_counter() - t0) * 1e3)
    n = len(arrs["feasible"])
    samples = int(arrs["n_samples"].sum())
    out["success_gate"] = {"trajectories": n, "samples": samples, "ms": float(np.median(t[1:])),
                           "trajectories_per_s": n / (float(np.median(t[1:])) * 1e-3),
                           "passed": int(arrs["feasible_print"].sum()), "winner": best,
                           "note": "checkFeasible + printConstraintsSituations of every candidate of the last "
                                   "256-candidate solve from the solver's device buffers, verdicts to the host"}
    if not with_cpu:
        return out
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    # oracle: ROG ring on a bounded ring (203 x 203 x 43)
    small = tp.rog_desc(half_prob_map_size_i=(100, 100, 20), local_update_box=(10.0, 10.0, 2.0))
    orc = O.RogField(small)
    p2 = pts[(np.abs(pts[:, 0]) < 4.9) & (np.abs(pts[:, 1]) < 4.9) & (pts[:, 2] < 0.95)]
    orc.update_counters(p2, np.full(len(p2), 1), np.full(len(p2), 3))
    t0 = time.perf_counter()
    orc.update_esdf((0.0, 0.0, 0.0))
    dt = time.perf_counter() - t0
    bvox = int(np.prod([2 * h for h in orc.half_box]))
    out["rog_update"]["cpu"] = {"Mvoxel_per_s": bvox / dt / 1e6, "ms": dt * 1e3, "cores": 1, "kind": "port",
                                "sample": f"ring {orc.size}, update box {bvox} voxels"}
    # oracle: ProbMap ingest of a 10^4-point frame on the bounded ring
    opm = O.RogProb(orc, small, tp.prob_desc(ray_range=(0.3, 10.0), virtual_ceil_height=3.0, virtual_ground_height=-0.5,
                                             local_update_box=(20.0, 20.0, 4.0), inflation_resolution=res))
    opm.update(cloud[:10000], (0.0, 0.0, 1.0))
    t0 = time.perf_counter()
    opm.update(cloud[10000:20000], (0.02, 0.0, 1.0))
    dt = time.perf_counter() - t0
    out["prob_map_update"]["cpu"] = {"Mpoints_per_s": 0.01 / dt, "ms": dt * 1e3, "cores": 1, "kind": "port",
                                     "sample": f"10^4 points on ring {orc.size} (incl. updateESDF3D)"}
    # oracle: dense field rebuild + queries at the default 200 x 200 x 16 grid
    desc = tp.grid_desc()
    of = O.Field(desc)
    spts, _ = scenes.cuboids_scene(42)
    of.rasterize(spts)
    t0 = time.perf_counter()
    of.rebuild()
    dt = time.perf_counter() - t0
    ms_g = []
    for _ in range(4):
        gm.updateESDF()
        ms_g.append(gm.last_rebuild_ms()[0])
    q = np.concatenate([rng.uniform(-9.9, 9.9, (200000, 2)), rng.uniform(0.01, 1.59, (200000, 1))], axis=1)
    t0 = time.perf_counter()
    of.query3d(q)
    dq = time.perf_counter() - t0
    out["field_default_grid"] = {"grid": "200x200x16 @0.1 m (4 x 2-D maps + 3-D)", "gpu_rebuild_ms": float(np.median(ms_g[1:])),
                                 "cpu": {"rebuild_ms": dt * 1e3, "query_Mpoints_per_s": len(q) / dq / 1e6, "cores": 1,
                                         "kind": "port", "sample": "one rebuild; 2e5 value+gradient queries"}}
    # oracle: the gate on 8 of the solved trajectories
    trajs = [solver.getTraj(c)._tuple() for c in range(min(8, n))]
    t0 = time.perf_counter()
    O.check_feasible(of, rp, trajs)
    dt = time.perf_counter() - t0
    out["success_gate"]["cpu"] = {"trajectories_per_s": len(trajs) / dt, "cores": 1, "kind": "port",
                                  "sample": f"{len(trajs)} of the solved trajectories, {dt:.2f} s"}
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, res, first, n):
    """--dump-outputs: what MomaTrajOpt.download() hands a caller for candidates first .. first + n - 1 (the last
    plan of the timed solve), one float64 DIR/<name>.npy per result array, candidates along the first axis. Above
    64 MB in all, a fixed seeded sample of the candidates is written. candidate_index.npy lists the candidates
    written (index inside the plan)."""
    rows = {k: v[first:first + n] for k, v in res.items() if isinstance(v, np.ndarray)}
    per_cand = 8 * (1 + sum(v[0].size for v in rows.values()))
    m = min(n, (DUMP_BYTES - 4096 * (len(rows) + 1)) // per_cand)
    idx = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "candidate_index.npy"), idx.astype(np.float64))
    for k, v in rows.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v[idx].astype(np.float64))


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for the path on the host cores — the oracle port (bit-identical
    to the reference's optimizer and map compiled unmodified, tests/test_ref_pin.py); rank 0
    alone runs it. (See CpuArm for why the timed arm is the port unless TOPAY_BENCH_CPU_REF=1.)"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import topay_b200._structs as S  # structs only; no GPU library needed on this arm
    from topay_b200 import scenes
    desc = S.grid_desc()
    pts, _ = scenes.cuboids_scene(42)
    arm = CpuArm(desc, pts)
    opt = arm.O.opt_defaults()
    opt.int_K, opt.min_piece_num, opt.sample_interval = INT_K, N_PIECES, 1e9
    cores = os.cpu_count() or 1
    paths, bv, ba = scenes.synthetic_batch(N_CAND, 1234)
    m = min(cores, N_CAND)
    warm = min(args.warmup, 1)     # warm-up passes actually run: a CPU solve needs no clock/cache warm-up beyond one
    step_i = 0

    def one_step():
        nonlocal step_i
        lo = (step_i * m) % (N_CAND - m + 1)     # a different slice of the batch every step
        step_i += 1
        return arm.solve_batch(opt, paths[lo:lo + m], bv[lo:lo + m], ba[lo:lo + m], cores)

    for _ in range(warm):
        one_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_step()
    dt = time.perf_counter() - t0
    value = m * args.steps / dt
    line = {
        "impl": "reference", "metric": "optimized trajectories/sec at 256 candidates", "value": value,
        "unit": "trajectories/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "warmup_passes_run": warm,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": base_config(N_CAND),
        "cpu_baseline": {"value": value, "unit": "trajectories/s", "cores": cores, "kind": arm.kind,
                         "sample": f"{m} of the {N_CAND} candidates per step (one per host core, thread per "
                                   f"candidate), a different slice each step"},
        "e2e": {"value": value, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="topay_b200", choices=["topay_b200", "reference"])
    ap.add_argument("--candidates", type=int, default=N_CAND, help="candidates per plan (dev only; bench = 256)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (dev only)")
    ap.add_argument("--no-extras", action="store_true", help="skip the latency and field sub-benchmarks")
    ap.add_argument("--slots", type=int, default=2048,
                    help="candidates in flight on the device (continuous batching: a finished candidate's slot is "
                         "refilled from the queue of waiting plans on the device)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed plan to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device solve's results; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local, dist = dist_setup(args.gpus)
    import torch
    import topay_b200 as tp
    from topay_b200 import scenes
    torch.cuda.set_device(local)
    n_cand = args.candidates
    opt, rp = workload_params(tp)
    desc = tp.grid_desc()
    pts, _ = scenes.cuboids_scene(42)
    gm = tp.GridMap(desc, device=local)
    gm.regenerateMap(pts)
    K, W = args.steps, max(args.warmup, 0)
    # One step = one plan of 256 candidates. Every rank owns DISTINCT plans (seeded by rank and step): candidates
    # and plans are independent, so they shard with no data-path collective (weak scaling: K plans per GPU). The
    # K plans of a rank are queued on its device and stream through a fixed pool of candidate slots.
    plans = [scenes.synthetic_batch(n_cand, 1234 + 1000 * (rank * K + p)) for p in range(K)]
    paths, bv, ba = plans[0]
    n_slots = max(1, min(args.slots, K * n_cand))
    solver = tp.MomaTrajOpt(gm, max_cand=K * n_cand, max_pieces=N_PIECES, opt_param=opt, robot=rp, n_slots=n_slots)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=f"cuda:{local}")   # > 126 MB L2

    def cat(pl):
        return ([q for p in pl for q in p[0]], np.concatenate([p[1] for p in pl]), np.concatenate([p[2] for p in pl]))

    # ---- warm-up: W plans through the pool (graphs instantiated, clocks up)
    if W > 0:
        solver.upload(*cat([plans[i % K] for i in range(W)]))
        solver.run()
    # ---- resident arm: the K plans pre-processed and uploaded once, one timed device solve of all of them
    solver.upload(*cat(plans))
    torch.cuda.synchronize()
    barrier_max(dist, local, 0.0)
    sampler = ClockSampler(local) if rank == 0 else None
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    solver.run()
    torch.cuda.synchronize()
    dt = barrier_max(dist, local, time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None
    st_run = solver.stats()
    res = solver.download()
    n_ok = int(res["status"].sum())
    evals_total = int(res["evals"].sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, (K - 1) * n_cand, n_cand)

    # ---- end-to-end arm: host buffers in, host results out, through the public API — the worker flow of
    # planner.cpp:847-1010 (pre-processing, H2D of the problems, the solve, the success gate, the per-plan selection
    # and the D2H of each plan's winning trajectory inside the timed region)
    barrier_max(dist, local, 0.0)
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r_e2e = solver.planWinners(plans, use_gate=True)
    torch.cuda.synchronize()
    dt_e2e = barrier_max(dist, local, time.perf_counter() - t0)
    h2d, d2h = solver.h2d_bytes, solver.d2h_bytes

    # ---- BASELINE configs[4], bounded: independent scenarios sharded round-robin over the ranks (all ranks take part)
    sweep = None if args.no_extras else sweep_probe(tp, scenes, local, rank, world, dist)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline pass (rank 0, after the timed regions): the same pool on 4 plans with plain launches and CUDA
    # events around every kernel launch -> live per-kernel device time, averaged over the launches of the pass
    kr = min(K, 4)
    solver.upload(*cat(plans[:kr]))
    solver.set_timed(True)
    flush.zero_()
    solver.run()
    rst = solver.stats()
    solver.set_timed(False)
    # one plan alone (256 candidates, no refill): the tail-bound figure
    solver.upload(*plans[0])
    solver.run()
    t0 = time.perf_counter()
    solver.run()
    dt_single = time.perf_counter() - t0
    st_single = solver.stats()

    total = n_cand * K * world
    value = total / dt
    peak, peak_src = measured_peaks()
    ticks_r = max(rst["ticks"], 1)
    k_ms = {"k_penalty": rst["ms_eval"], "k_cand<lbfgs>": rst["ms_lbfgs"], "k_cand<generate>": rst["ms_gen"],
            "k_cand<adjoint>": rst["ms_adj"], "k_chain": rst["ms_chain"], "k_integrate": rst["ms_integrate"]}
    k_sum = max(sum(k_ms.values()), 1e-9)
    shares = {k: v / k_sum for k, v in k_ms.items()}
    live_avg = rst["slot_ticks"] / ticks_r
    # k_cand<lbfgs>: algorithmic bytes = the L-BFGS history the two-loop recursions walk, counted on the device
    lb_ms = max(rst["ms_lbfgs"] / ticks_r, 1e-9)
    lb_bytes = rst["hist_bytes"] / ticks_r
    lb_achieved = lb_bytes / (lb_ms * 1e-3) / 1e9
    # k_penalty: 800 B of ESDF taps and 4.0 kflop per penalty node (SURVEY §8d)
    pen_ms = max(rst["ms_eval"] / ticks_r, 1e-9)
    nodes_per_launch = rst["eval_nodes"] / ticks_r
    pen_bytes = nodes_per_launch * NODE_BYTES
    pen_achieved = pen_bytes / (pen_ms * 1e-3) / 1e9
    flop = nodes_per_launch * NODE_FLOP + nodes_per_launch * INT_K / (INT_K + 1) * MID_FLOP
    roof_pen = {"bound": "hbm", "kernel": "k_penalty", "achieved": pen_achieved, "peak": peak, "unit": "GB/s",
                "frac": pen_achieved / peak, "traffic": 127.6e6,
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one mid-run launch with 1024 live "
                                  "candidates (2.16 M nodes, 1.73 GB algorithmic), ncu --set full, "
                                  "profiles/r02_summary.md section 4: the 5 MB field stays in L2",
                "peak_source": peak_src,
                "avg_launch_ms": pen_ms, "nodes_per_launch": nodes_per_launch,
                "algorithmic_bytes_per_launch": pen_bytes,
                "algorithmic_bytes": "800 B of ESDF taps per penalty node (12 x 3-D + 1 x 2-D lookups, SURVEY §8d) x the "
                                     "nodes of the live candidates of a launch; the 5 MB field is L2-resident, so the "
                                     "kernel is FP64-issue bound, not HBM bound (see fp64)",
                "share_of_step": shares["k_penalty"],
                "fp64": {"achieved_tflops": flop / (pen_ms * 1e-3) / 1e12, "nominal_peak_tflops": 40.0,
                         "note": "4.0 kflop per penalty node + 0.15 kflop per midpoint (SURVEY §8d); MEASURED_PEAKS.json "
                                 "has no FP64 figure, 40 TFLOP/s is the nominal B200 FP64 rate"}}
    roof_lb = {"bound": "hbm", "kernel": "k_cand<lbfgs>", "achieved": lb_achieved, "peak": peak, "unit": "GB/s",
               "frac": lb_achieved / peak, "traffic": 3.455e9,
               "traffic_source": "dram bytes of one mid-solve launch with 1024 live candidates in 0.60 ms (5.7 TB/s, "
                                 "gpu__dram_throughput 70.5 % of peak), ncu --set full, profiles/r02_summary.md section 4",
               "peak_source": peak_src, "avg_launch_ms": lb_ms,
               "algorithmic_bytes_per_launch": lb_bytes,
               "algorithmic_bytes": "L-BFGS history walked by the two-loop recursions: 2 loops x bound rows x (s_j, y_j) "
                                    "x n x 8 B per accepted iteration (5.2 MB at m = 256, n = 632), counted on the device; "
                                    "candidates in a line-search trial stream nothing",
               "share_of_step": shares["k_cand<lbfgs>"]}
    dominant = max(shares, key=shares.get)
    roofline = dict(roof_pen if dominant == "k_penalty" else roof_lb)
    roofline["kernel_shares"] = shares
    roofline["measured_on"] = (f"{kr} plans ({kr * n_cand} candidates) through the same {n_slots}-slot pool right after the "
                               f"timed regions, plain launches with CUDA events around every kernel launch; averages over "
                               f"all {rst['ticks']} ticks of the pass ({live_avg:.0f} live candidates per launch on average)")
    line = {
        "metric": "optimized trajectories/sec at 256 candidates", "value": value, "unit": "trajectories/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * dt / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(n_cand),
        "details": {"scheduling": f"continuous batching: the K plans of a rank ({K} x {n_cand} candidates, distinct per "
                                  f"rank and step) are queued on the device and stream through {n_slots} candidate "
                                  f"slots; a finished candidate's slot takes the next waiting candidate inside the kernel; pools of 512+ "
                                  f"slots run as two lanes (two parallel branches of the tick graph) so that one half's "
                                  f"FP64-bound penalty kernel overlaps the other half's HBM- / latency-bound L-BFGS kernels",
                    "slots": n_slots,
                    "l2": f"working set larger than L2: the L-BFGS history is 2.6 MB per slot ({2.6e-3 * n_slots:.1f} GB at "
                          f"{n_slots} slots, 126 MB L2); a 512 MiB buffer is rewritten before each timed region",
                    "successes": n_ok},
        "e2e": {"value": total / dt_e2e, "unit": "trajectories/s", "h2d_bytes_per_step": h2d // K,
                "d2h_bytes_per_step": d2h // K,
                "plans_with_a_feasible_winner": int(sum(w is not None for w in r_e2e)),
                "api": "MomaTrajOpt.planWinners(plans): host waypoints -> pre-processing -> pinned H2D -> device solve "
                       "of every candidate -> success gate (checkFeasible / printConstraintsSituations) and "
                       "shortest-duration selection per plan on the device -> D2H of the gate's per-trajectory "
                       "metrics and of each plan's winning trajectory (status, cost, durations, coefficients, x)"},
        "gpu_launches": int(st_run["kernel_launches"]),
        "device_ms_per_step": st_run["ms_total"] / K, "ticks": int(st_run["ticks"]),
        "slot_utilisation": evals_total / max(st_run["slot_ticks"], 1),
        "evals_per_candidate": evals_total / max(n_cand * K, 1),
        "us_per_evaluation": 1e3 * st_run["ms_total"] / max(evals_total, 1),
        "single_plan": {"value": n_cand / dt_single, "unit": "trajectories/s", "ms": dt_single * 1e3,
                        "ticks": int(st_single["ticks"]),
                        "note": "one 256-candidate plan alone on the device (no other plan to refill from): bound by "
                                "its slowest candidate"},
        "roofline": roofline,
        "roofline_k_penalty": roof_pen,
        "roofline_k_lbfgs": roof_lb,
        "clocks": clocks,
    }
    if sweep is not None:
        line["sweep"] = sweep
    if not args.no_extras and world == 1:     # single-GPU diagnostics; the scaling runs stay short
        line["latency"] = latency_probe(tp, scenes, gm)
        line["field"] = field_probe(tp, scenes, local, peak)
        line["field"]["solve_on_this_field"]["k_penalty_ns_per_node_on_the_5MB_field"] = 1e6 * pen_ms / max(nodes_per_launch, 1)
        solver.upload(*plans[0])
        solver.run()
        solver.download()
        line["subpaths"] = subpath_probe(tp, scenes, local, peak, solver, gm, rp, not args.no_cpu_baseline)
    if not args.no_cpu_baseline and world == 1:   # rank 0 at N = 1 only
        cores = os.cpu_count() or 1
        line["cpu_baseline"] = cpu_baseline(opt, rp, pts, paths, bv, ba, cores, desc)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
