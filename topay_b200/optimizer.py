"""MomaTrajOpt — host-side mirror of the reference's trajectory optimizer over the C ABI.

nmoma_planner::MomaTrajOpt (src/planner/include/planner/moma_traj_opt.h:613-675) is one
single-threaded instance per candidate; the reference runs up to 8 of them on threads
(planner.cpp:59-66, 921-925). Here one object owns the device state for a whole batch:
`optimizeTraj` keeps the reference's call shape for one candidate, `optimizeTrajBatch` is the
batched entry the planner's worker pool collapses into.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._structs import (NTERMS, OptParams, ProblemBatch, ResultBatch, RobotParams, SolverStats, alloc_feasibility,
                       num_vars, pack_trajs)
from .field import GridMap, _p, robot_params_default


def opt_params_default():
    o = OptParams()
    _lib.lib().topay_opt_params_default(C.byref(o))
    return o


class MomaTraj:
    """Result of one optimisation (moma_traj_opt.h:26-247): piece durations + MINCO coefficients (row 6i+k =
    t^k of piece i, columns theta, arc, q1..q7 — MinJerkOpt<9>::getCoeffs layout, minco.hpp:944) + the SE(2)
    start. The pose table and the state samplers are evaluated on the device."""

    def __init__(self, T, coeff, start_se2, device=0):
        self.durations = np.ascontiguousarray(T, dtype=np.float64)
        self.coeff = np.ascontiguousarray(coeff, dtype=np.float64).reshape(6 * len(self.durations), 9)
        self.start_se2 = np.ascontiguousarray(start_se2, dtype=np.float64)[:3]
        self.device = device
        self.is_init = True
        self._car_seq = None

    def _tuple(self):
        return (self.durations, self.coeff, self.start_se2)

    def getTotalDuration(self):
        return float(sum(float(t) for t in self.durations))     # summed in piece order (minco.hpp:304-313)

    @property
    def car_seq(self):
        """(m, 4) rows x, y, yaw, t every seq_res = 0.1 s (moma_traj_opt.h:38-68)."""
        if self._car_seq is None:
            tb, keep = pack_trajs([self._tuple()])
            cap = int(self.getTotalDuration() / 0.1) + 4
            out = np.zeros((1, cap, 4))
            ln = np.zeros(1, dtype=np.int32)
            _lib.check(_lib.lib().topay_traj_car_seq(self.device, C.byref(tb), cap, _p(out), _p(ln, C.c_int32)),
                       "topay_traj_car_seq")
            self._car_seq = out[0, :ln[0]].copy()
        return self._car_seq

    def _sample(self, t, want_state=True, want_dstate=False):
        t = np.ascontiguousarray(np.atleast_1d(t), dtype=np.float64).reshape(1, -1)
        tb, keep = pack_trajs([self._tuple()])
        st = np.zeros((1, t.shape[1], 10)) if want_state else None
        ds = np.zeros((1, t.shape[1], 10)) if want_dstate else None
        _lib.check(_lib.lib().topay_traj_sample(self.device, C.byref(tb), _p(t), t.shape[1], _p(st), _p(ds)),
                   "topay_traj_sample")
        return (st[0] if want_state else None), (ds[0] if want_dstate else None)

    def getState(self, t):
        """MomaTraj::getState (moma_traj_opt.h:121-149): (x, y, yaw, q1..q7) at one time or an array of times."""
        st = self._sample(t)[0]
        return st[0] if np.ndim(t) == 0 else st

    def getDState(self, t):
        """MomaTraj::getDState (moma_traj_opt.h:151-160): (v, omega, 0, dq1..dq7)."""
        ds = self._sample(t, want_state=False, want_dstate=True)[1]
        return ds[0] if np.ndim(t) == 0 else ds

    @staticmethod
    def normYaw(yaw):
        y = np.array(yaw, dtype=np.float64)
        while np.any(y > np.pi):
            y = np.where(y > np.pi, y - 2 * np.pi, y)
        while np.any(y < -np.pi):
            y = np.where(y < -np.pi, y + 2 * np.pi, y)
        return y

    def sampleTimePoints(self, n):
        """moma_traj_opt.h:172-199: n rows (x, y, yaw normalised, q1..q7, cos yaw, sin yaw) at equal time steps."""
        num = n - 2
        total = self.getTotalDuration()
        dt = total / (num + 1)
        t = np.array([i * dt for i in range(num + 1)] + [total])
        x = self.getState(t)
        x[:, 2] = self.normYaw(x[:, 2])
        return np.concatenate([x, np.cos(x[:, 2:3]), np.sin(x[:, 2:3])], axis=1)


class MomaTrajOpt:
    def __init__(self, grid_map: GridMap, max_cand=8, max_pieces=16, opt_param: OptParams = None,
                 robot: RobotParams = None, n_slots=None):
        """max_cand: candidates one upload may hold (several plans back to back); n_slots: how many of them are in
        flight on the device at a time (default: all) — finished candidates hand their slot to the next waiting
        one on the device (topay_solver_create_pool)."""
        self._l = _lib.lib()
        self.grid_map = grid_map
        self.opt_param = opt_param if opt_param is not None else opt_params_default()
        self.moma_param = robot if robot is not None else robot_params_default()
        self.max_cand, self.max_pieces = max_cand, max_pieces
        self.h = C.c_void_p()
        # GridMap::use_rog (grid_map.h:90): a rog.ESDFMap routes every field lookup of the solve and of the gate
        # to the ROG-Map ring
        self.use_rog = not isinstance(grid_map, GridMap)
        self.n_slots = max_cand if n_slots is None else min(n_slots, max_cand)
        if self.use_rog or self.n_slots == max_cand:
            create = self._l.topay_solver_create_rog if self.use_rog else self._l.topay_solver_create
            _lib.check(create(C.byref(self.opt_param), C.byref(self.moma_param), grid_map.h, max_cand, max_pieces,
                              C.byref(self.h)), "topay_solver_create")
        else:
            _lib.check(self._l.topay_solver_create_pool(C.byref(self.opt_param), C.byref(self.moma_param), grid_map.h,
                                                        max_cand, self.n_slots, max_pieces, C.byref(self.h)),
                       "topay_solver_create_pool")
        self.traj_cost = 0.0
        self._last = None
        self._stream = {}      # streaming session: plan id -> (candidates, start poses, field kept alive)

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self._l.topay_solver_destroy(self.h)
            self.h = C.c_void_p()

    __del__ = close

    # ---- parity hook: one cost/gradient evaluation per candidate ---------------
    def evaluate(self, stage, piece_num, head_pva, tail_pva, start_xy, end_xy, init_inner_xy, x, alm_lambda=None,
                 alm_rho=None):
        """firstStageCostCallback / secondStageCostCallback (moma_traj_opt.cpp:817-955) for a batch.
        x: (n, num_vars(max_pieces)) padded. Returns dict(cost, grad, terms, coeff, final_xy)."""
        n = len(piece_num)
        NP = self.max_pieces
        xs = num_vars(NP)
        pn = np.ascontiguousarray(piece_num, dtype=np.int32)
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (head_pva, tail_pva, start_xy, end_xy)]
        ixy = np.zeros((n, NP, 2))
        for c in range(n):
            ixy[c, :pn[c]] = np.asarray(init_inner_xy[c])[:pn[c]]
        lam = np.ascontiguousarray(alm_lambda if alm_lambda is not None else np.zeros((n, 2)), dtype=np.float64)
        rho = np.ascontiguousarray(alm_rho if alm_rho is not None else np.ones((n, 2)), dtype=np.float64)
        xb = np.zeros((n, xs))
        for c in range(n):
            xb[c, :num_vars(pn[c])] = np.asarray(x[c])[:num_vars(pn[c])]
        pb = ProblemBatch(n, _p(pn, C.c_int32), _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), _p(ixy), _p(lam),
                          _p(rho))
        cost, grad = np.zeros(n), np.zeros((n, xs))
        terms, coeff, fxy = np.zeros((n, NTERMS)), np.zeros((n, 6 * NP, 9)), np.zeros((n, 2))
        _lib.check(self._l.topay_solver_eval(self.h, stage, C.byref(pb), _p(xb), xs, _p(cost), _p(grad), _p(terms),
                                             _p(coeff), _p(fxy)), "topay_solver_eval")
        return dict(cost=cost, grad=grad, terms=terms, coeff=coeff, final_xy=fxy)

    # ---- solve -------------------------------------------------------------------
    def _flatten(self, paths, bvel, bacc):
        n = len(paths)
        plen = np.array([np.asarray(p).shape[0] for p in paths], dtype=np.int32)
        flat = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.float64) for p in paths], axis=0))
        bvel = np.ascontiguousarray(bvel, dtype=np.float64).reshape(n, 10, 2)
        bacc = np.ascontiguousarray(bacc, dtype=np.float64).reshape(n, 10, 2)
        return n, plen, flat, bvel, bacc

    def upload(self, paths, bvel, bacc):
        n, plen, flat, bvel, bacc = self._flatten(paths, bvel, bacc)
        _lib.check(self._l.topay_solver_upload(self.h, n, _p(plen, C.c_int32), _p(flat), _p(bvel), _p(bacc)),
                   "topay_solver_upload")
        self._n = n
        self._starts = [np.asarray(p)[0, :3].copy() for p in paths]
        self.h2d_bytes = int(plen.nbytes + flat.nbytes + bvel.nbytes + bacc.nbytes)

    def assign_fields(self, fields, field_of):
        """topay_solver_assign_fields: candidate c of the uploaded batch is solved (and gated) against fields[field_of[c]]
        — scenario sweeps, where one upload carries the candidates of many scenarios. `fields` = GridMap objects on
        this solver's device, rebuilt before run(); None / a single field returns to the solver's own field."""
        if not fields or len(fields) <= 1:
            _lib.check(self._l.topay_solver_assign_fields(self.h, None, 0, None), "topay_solver_assign_fields")
            self._fields = None
            return
        hs = (C.c_void_p * len(fields))(*[f.h for f in fields])
        fo = np.ascontiguousarray(field_of, dtype=np.int32)
        assert len(fo) == self._n
        _lib.check(self._l.topay_solver_assign_fields(self.h, hs, len(fields), _p(fo, C.c_int32)), "topay_solver_assign_fields")
        self._fields = list(fields)       # keep them alive

    def set_plans(self, plan_offset=None, grace_evals=None, use_gate=False):
        """topay_solver_set_plans: first success + grace of the planner's worker pool (planner.cpp:931-952), counted
        in evaluations. plan_offset: first candidate of each plan + the total (default: one plan = the whole upload).
        Once a plan has a success (status 1 and, with use_gate, printConstraintsSituations), its candidates that need
        more than grace_evals evaluations beyond that success's are cancelled (status 0, lbfgs_code
        LBFGSERR_PLAN_GRACE, results zero); the others are bit-identical to a run without plans. grace_evals=None
        turns it off. The setting holds for uploads of the same size until it is changed."""
        if grace_evals is None:
            _lib.check(self._l.topay_solver_set_plans(self.h, 0, None, 0, 0), "topay_solver_set_plans")
            return
        off = np.ascontiguousarray([0, self._n] if plan_offset is None else plan_offset, dtype=np.int32)
        _lib.check(self._l.topay_solver_set_plans(self.h, len(off) - 1, _p(off, C.c_int32), int(use_gate),
                                                  int(grace_evals)), "topay_solver_set_plans")

    def run(self):
        _lib.check(self._l.topay_solver_run(self.h), "topay_solver_run")

    def _result_arrays(self, n):
        """Result arrays for n candidates and the ResultBatch that points the library at them."""
        NP = self.max_pieces
        r = dict(status=np.zeros(n, np.int32), lbfgs_code=np.zeros(n, np.int32), piece_num=np.zeros(n, np.int32),
                 iters=np.zeros(n, np.int32), evals=np.zeros(n, np.int32), alm_rounds=np.zeros(n, np.int32),
                 cost=np.zeros(n), duration=np.zeros(n), T=np.zeros((n, NP)), coeff=np.zeros((n, 6 * NP, 9)),
                 final_xy_err=np.zeros((n, 2)), x=np.zeros((n, num_vars(NP))))
        rb = ResultBatch(*[_p(r[k], C.c_int32 if r[k].dtype == np.int32 else C.c_double) for k in
                           ("status", "lbfgs_code", "piece_num", "iters", "evals", "alm_rounds", "cost", "duration",
                            "T", "coeff", "final_xy_err", "x")])
        return r, rb

    def download(self):
        r, rb = self._result_arrays(self._n)
        bd, bc = C.c_int32(-1), C.c_int32(-1)
        _lib.check(self._l.topay_solver_download(self.h, C.byref(rb), C.byref(bd), C.byref(bc)), "download")
        r["best_by_duration"], r["best_by_cost"] = bd.value, bc.value
        self.d2h_bytes = int(sum(v.nbytes for v in r.values() if isinstance(v, np.ndarray)))
        self._last = r
        return r

    def select(self, plan_offset=None, use_gate=False):
        """topay_solver_select: the planner's pick (planner.cpp:999-1010) per plan ON THE DEVICE; two ints per plan
        come back. plan_offset: first candidate of each plan + the total (default: one plan = the whole upload).
        Returns (best_by_duration, best_by_cost): indices inside each plan, -1 where no candidate qualifies."""
        off = np.ascontiguousarray([0, self._n] if plan_offset is None else plan_offset, dtype=np.int32)
        n_plans = len(off) - 1
        bd, bc = np.full(n_plans, -1, np.int32), np.full(n_plans, -1, np.int32)
        _lib.check(self._l.topay_solver_select(self.h, n_plans, _p(off, C.c_int32), int(use_gate), _p(bd, C.c_int32),
                                               _p(bc, C.c_int32)), "topay_solver_select")
        return bd, bc

    def download_candidate(self, cand):
        """Results of one candidate of the last run (the winner): 28 KB at 64 pieces instead of the whole batch."""
        r, rb = self._result_arrays(1)
        _lib.check(self._l.topay_solver_download_candidate(self.h, int(cand), C.byref(rb)), "download_candidate")
        out = {k: v[0] for k, v in r.items()}
        out["index"] = int(cand)
        out["nbytes"] = int(sum(v.nbytes for v in r.values()))
        return out

    def planWinners(self, plans, use_gate=True, fields=None, grace_evals=None):
        """The worker loop of planner.cpp:847-1010 for several plans in one device solve: every candidate is optimised
        (continuous batching), passed through the success gate (optimizeTraj && printConstraintsSituations,
        :877-880) and the shortest trajectory of each plan is picked (:999-1010) — all on the device; only each
        plan's winner crosses the bus. Returns a list with one entry per plan: the winner's result dict
        (download_candidate, `index` inside the plan) or None. `fields`: one GridMap per plan (scenario sweeps: every
        plan is solved and gated against its own scenario's field, all plans share the launches of one solve).
        grace_evals: first success + grace per plan (set_plans; None = off)."""
        paths = [q for p in plans for q in p[0]]
        bv = np.concatenate([np.asarray(p[1], dtype=np.float64).reshape(len(p[0]), 10, 2) for p in plans])
        ba = np.concatenate([np.asarray(p[2], dtype=np.float64).reshape(len(p[0]), 10, 2) for p in plans])
        self.upload(paths, bv, ba)
        if fields is not None:      # plan i against its own scenario's field (scenario sweeps)
            self.assign_fields(fields, np.repeat(np.arange(len(plans)), [len(p[0]) for p in plans]))
        off = np.cumsum([0] + [len(p[0]) for p in plans]).astype(np.int32)
        self.set_plans(off, grace_evals, use_gate)
        self.run()
        self.d2h_bytes = 0
        if use_gate:
            f, arrs = alloc_feasibility(self._n, verdicts_only=True)
            _lib.check(self._l.topay_solver_check_feasible(self.h, C.byref(f), None), "topay_solver_check_feasible")
            self.constraints = arrs
            self.d2h_bytes += self._n * 352     # what the gate itself reads back: per-trajectory metrics + sizes
        bd, _ = self.select(off, use_gate)
        self.d2h_bytes += int(bd.nbytes * 2)
        out = []
        for i, w in enumerate(bd):
            if w < 0:
                out.append(None)
                continue
            r = self.download_candidate(int(off[i] + w))
            r["index"] = int(w)
            self.d2h_bytes += r["nbytes"]
            out.append(r)
        self._last = None
        return out

    # ---- streaming session: plans arrive while the solve runs ------------------------
    def stream_begin(self, use_gate=False, grace_evals=None, snapshots=0):
        """topay_solver_stream_begin: from here on plans are submitted while the solve runs and each plan's winners
        come back as soon as its last candidate has finished. use_gate: winners must pass printConstraintsSituations.
        grace_evals: first success + grace for every plan of the session (stream_set_grace; None = off). snapshots:
        ring snapshots of a ROG solver (stream_set_snapshots; 0 = off). The uploaded batch is dropped; the batch calls
        are refused until stream_end()."""
        _lib.check(self._l.topay_solver_stream_begin(self.h, int(use_gate)), "topay_solver_stream_begin")
        self._stream = {}
        if grace_evals is not None:
            self.stream_set_grace(grace_evals)
        if snapshots:
            self.stream_set_snapshots(snapshots)

    def stream_set_snapshots(self, n):
        """topay_solver_stream_set_snapshots (ROG solver): n >= 1 pins every plan submitted from now on to a copy of the
        ring as it is at the submit, so the map may slide and update while plans solve; each plan is bit-identical to
        its solo batch solve on the ring of its submit (ring updates come from this solver's thread, or are serialised
        with its calls). Up to n ring states are held at once by untaken plans (a
        submit that needs one more is refused with TOO_LARGE). 0 = plans read the live ring. Refused (NOT_READY)
        while a submitted plan has not been taken."""
        _lib.check(self._l.topay_solver_stream_set_snapshots(self.h, int(n)), "topay_solver_stream_set_snapshots")

    def stream_set_grace(self, grace_evals=None):
        """topay_solver_stream_set_grace: first success + grace (set_plans) for every plan streamed from now on; each
        is bit-identical to its solo batch solve with that grace. None turns it off. Refused (NOT_READY) while a
        submitted plan has not finished."""
        _lib.check(self._l.topay_solver_stream_set_grace(self.h, -1 if grace_evals is None else int(grace_evals)),
                   "topay_solver_stream_set_grace")

    def stream_stop(self, plan_id):
        """topay_solver_stream_stop: cancels the live plan's remaining candidates (the reference's interrupt_all); the
        plan is then reported by stream_poll as usual, its winners taken from the candidates that finished before the
        stop. A finished plan is left as it is."""
        _lib.check(self._l.topay_solver_stream_stop(self.h, int(plan_id)), "topay_solver_stream_stop")

    def stream_submit(self, paths, bvel, bacc, field=None):
        """Queues one plan (its candidates' waypoint lists and boundary velocities / accelerations, as upload()) and
        returns its plan id. field: the GridMap the plan is solved and gated against (None: the solver's own)."""
        n, plen, flat, bvel, bacc = self._flatten(paths, bvel, bacc)
        pid = C.c_int32(-1)
        _lib.check(self._l.topay_solver_stream_submit(self.h, n, _p(plen, C.c_int32), _p(flat), _p(bvel), _p(bacc),
                                                      field.h if field is not None else None, C.byref(pid)),
                   "topay_solver_stream_submit")
        self._stream[pid.value] = (n, [np.asarray(p)[0, :3].copy() for p in paths], field)
        return pid.value

    def stream_advance(self, max_batches=1):
        """Runs up to max_batches batches of 16 ticks; returns the candidates still in the slots (0: all done)."""
        live = C.c_int32(0)
        _lib.check(self._l.topay_solver_stream_advance(self.h, int(max_batches), C.byref(live)),
                   "topay_solver_stream_advance")
        return live.value

    def stream_poll(self, cap=None):
        """Finished plans not reported before: a list of (plan_id, best_by_duration, best_by_cost), winners as
        indices inside the plan (-1: none)."""
        cap = self.max_cand if cap is None else int(cap)
        pid, bd, bc = (np.full(max(cap, 1), -1, np.int32) for _ in range(3))
        k = self._l.topay_solver_stream_poll(self.h, cap, _p(pid, C.c_int32), _p(bd, C.c_int32), _p(bc, C.c_int32))
        if k < 0:
            _lib.check(k, "topay_solver_stream_poll")
        return [(int(pid[i]), int(bd[i]), int(bc[i])) for i in range(k)]

    def stream_take(self, plan_id, cand=None, gate=False):
        """Results of a finished plan, then its rows and id are free: the dict of download() over its candidates, or
        with `cand` the dict of download_candidate() for that one. gate=True adds the gate metrics under "gate"."""
        n = self._stream[plan_id][0] if plan_id in self._stream else 1
        m = n if cand is None else 1
        r, rb = self._result_arrays(m)
        f, arrs = alloc_feasibility(m) if gate else (None, None)
        _lib.check(self._l.topay_solver_stream_take(self.h, int(plan_id), -1 if cand is None else int(cand),
                                                    C.byref(rb), C.byref(f) if gate else None),
                   "topay_solver_stream_take")
        starts = self._stream.pop(plan_id)[1]
        if cand is not None:
            r = {k: v[0] for k, v in r.items()}
            r["index"] = int(cand)
            if gate:
                arrs = {k: v[0] for k, v in arrs.items()}
        r["starts"] = starts if cand is None else starts[int(cand)]
        if gate:
            r["gate"] = arrs
        return r

    def stream_end(self):
        """Ends the session, dropping every plan not taken; the solver is back in batch mode."""
        _lib.check(self._l.topay_solver_stream_end(self.h), "topay_solver_stream_end")
        self._stream = {}

    def optimizeTrajBatch(self, paths, boundary_vel, boundary_acc, grace_evals=None):
        """All candidates of a plan in one device solve; returns the result dict of download(). grace_evals: first
        success + grace over the batch as one plan (set_plans; None = off)."""
        self.upload(paths, boundary_vel, boundary_acc)
        self.set_plans(None, grace_evals)
        self.run()
        return self.download()

    def optimizeTrajPlans(self, plans, grace_evals=None):
        """Several plans through one device solve with continuous batching: `plans` is a list of
        (paths, boundary_vel, boundary_acc); their candidates are queued back to back and flow through the solver's
        slots (n_slots in flight, the next waiting candidate takes a slot the moment one finishes). Returns the
        result dict of download() over all candidates plus `plan_offset` (first candidate of each plan) and the
        per-plan winners `plan_best_by_duration` / `plan_best_by_cost` (index inside the plan, -1 if none).
        grace_evals: first success + grace per plan (set_plans; None = off)."""
        paths = [q for p in plans for q in p[0]]
        bv = np.concatenate([np.asarray(p[1], dtype=np.float64).reshape(len(p[0]), 10, 2) for p in plans])
        ba = np.concatenate([np.asarray(p[2], dtype=np.float64).reshape(len(p[0]), 10, 2) for p in plans])
        self.upload(paths, bv, ba)
        off = np.cumsum([0] + [len(p[0]) for p in plans])
        self.set_plans(off, grace_evals)
        self.run()
        r = self.download()
        bd, bc = [], []
        for i in range(len(plans)):
            ok = np.flatnonzero(r["status"][off[i]:off[i + 1]] == 1)
            if len(ok) == 0:
                bd.append(-1)
                bc.append(-1)
                continue
            dur, cost = r["duration"][off[i]:off[i + 1]][ok], r["cost"][off[i]:off[i + 1]][ok]
            bd.append(int(ok[np.argmin(dur)]))      # argmin takes the first minimum: planner.cpp:999-1010
            bc.append(int(ok[np.argmin(cost)]))
        r["plan_offset"], r["plan_best_by_duration"], r["plan_best_by_cost"] = off, np.array(bd), np.array(bc)
        return r

    def optimizeTraj(self, init_path, boundary_vel, boundary_acc):
        """bool MomaTrajOpt::optimizeTraj(init_path, boundary_vel, boundary_acc) (moma_traj_opt.cpp:142)."""
        r = self.optimizeTrajBatch([init_path], np.asarray(boundary_vel)[None], np.asarray(boundary_acc)[None])
        self.traj_cost = float(r["cost"][0])
        return bool(r["status"][0])

    def getTraj(self, idx=0):
        r = self._last
        N = int(r["piece_num"][idx])
        return MomaTraj(r["T"][idx, :N].copy(), r["coeff"][idx, :6 * N].copy(), self._starts[idx],
                        device=self.grid_map.device)

    # ---- success gate (planner.cpp:877-880) --------------------------------------
    def checkFeasible(self, trajs):
        """bool MomaTrajOpt::checkFeasible(MomaTraj) (moma_traj_opt.h:948-1045) for one trajectory or a list;
        returns the verdict(s). The accumulated metrics of the last call are in self.constraints."""
        single = isinstance(trajs, MomaTraj)
        lst = [trajs] if single else list(trajs)
        tb, keep = pack_trajs([t._tuple() for t in lst])
        f, arrs = alloc_feasibility(len(lst))
        # on a ROG solver the ring as it is now: is the trajectory being executed still feasible on the updated map?
        check = self._l.topay_traj_check_feasible_rog if self.use_rog else self._l.topay_traj_check_feasible
        _lib.check(check(self.grid_map.h, C.byref(self.moma_param), C.byref(tb), C.byref(f)),
                   "topay_traj_check_feasible")
        self.constraints = arrs
        return bool(arrs["feasible"][0]) if single else arrs["feasible"].astype(bool)

    def printConstraintsSituations(self, trajs):
        """moma_traj_opt.h:1047-1210: the same scan; the manipulator clearances are reported, not enforced."""
        single = isinstance(trajs, MomaTraj)
        self.checkFeasible(trajs)
        v = self.constraints["feasible_print"].astype(bool)
        return bool(v[0]) if single else v

    def checkFeasibleBatch(self):
        """The gate for every candidate of the last solve without leaving the device: returns (metrics dict,
        index of the shortest candidate with status && printConstraintsSituations, or -1)."""
        f, arrs = alloc_feasibility(self._n)
        best = C.c_int32(-1)
        _lib.check(self._l.topay_solver_check_feasible(self.h, C.byref(f), C.byref(best)),
                   "topay_solver_check_feasible")
        self.constraints = arrs
        return arrs, best.value

    def set_timed(self, timed):
        """Per-launch CUDA-event timing of the penalty kernel (plain launches) instead of graph replay."""
        _lib.check(self._l.topay_solver_set_timed(self.h, int(timed)), "topay_solver_set_timed")

    def set_trace(self, cap):
        _lib.check(self._l.topay_solver_set_trace(self.h, cap), "topay_solver_set_trace")
        self._trace_cap = cap

    def trace(self, cand):
        """(m, 4) array: f, step, k, ls of every accepted L-BFGS iteration of candidate `cand`."""
        out = np.zeros((self._trace_cap, 4))
        n = C.c_int32()
        _lib.check(self._l.topay_solver_download_trace(self.h, cand, _p(out), self._trace_cap, C.byref(n)), "trace")
        return out[:n.value].copy()

    def stats(self):
        s = SolverStats()
        self._l.topay_solver_last_stats(self.h, C.byref(s))
        return {k: getattr(s, k) for k, _ in SolverStats._fields_}


def prepare_candidate(opt, rp, init_path, bvel, bacc, max_pieces):
    """topay_prepare_candidate: the host pre-processing of optimizeTraj (moma_traj_opt.cpp:146-344)."""
    init_path = np.ascontiguousarray(init_path, dtype=np.float64)
    bvel, bacc = np.ascontiguousarray(bvel, dtype=np.float64), np.ascontiguousarray(bacc, dtype=np.float64)
    N, past = C.c_int32(), C.c_int32()
    head, tail, sxy, exy = np.zeros((9, 3)), np.zeros((9, 3)), np.zeros(2), np.zeros(2)
    inner_xy, x0 = np.zeros((max_pieces, 2)), np.zeros(num_vars(max_pieces))
    rc = _lib.lib().topay_prepare_candidate(C.byref(opt), C.byref(rp), _p(init_path), init_path.shape[0], _p(bvel),
                                            _p(bacc), max_pieces, C.byref(N), _p(head), _p(tail), _p(sxy), _p(exy),
                                            _p(inner_xy), _p(x0), C.byref(past))
    return dict(rc=rc, piece_num=N.value, head_pva=head, tail_pva=tail, start_xy=sxy, end_xy=exy,
                init_inner_xy=inner_xy, x0=x0[:num_vars(N.value)] if rc == 0 else x0, s1_past=past.value)


def getDensePath(raw_path, step_size, start_yaw, end_yaw, v_max, w_max):
    """GraphSearch::getDensePath (graph_search.cpp:119-176) through topay_dense_path: (n, 2) raw waypoints -> rows
    (x, y, theta, dt). Host arithmetic (the call every planning worker makes before the sampler and the solve,
    planner.cpp:858)."""
    raw = np.ascontiguousarray(raw_path, dtype=np.float64).reshape(-1, 2)
    cap = 64
    while True:
        out = np.zeros((cap, 4))
        n = _lib.lib().topay_dense_path(_p(raw), raw.shape[0], step_size, start_yaw, end_yaw, v_max, w_max, _p(out), cap)
        if n < 0:
            _lib.check(n, "topay_dense_path")
        if n <= cap:
            return out[:n]
        cap = n


def discretizePath(path, pt_num):
    """TopologyPRM::discretizePath (topo_prm.cpp:472-506) through topay_discretize_path: pt_num points at equal
    arc-length spacing along an (n, 3) polyline. Host arithmetic."""
    path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 3)
    out = np.zeros((int(pt_num), 3))
    _lib.check(_lib.lib().topay_discretize_path(_p(path), path.shape[0], int(pt_num), _p(out)), "topay_discretize_path")
    return out


def pathLength(path):
    """TopologyPRM::pathLength (topo_prm.cpp:462-470)."""
    path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 3)
    return float(_lib.lib().topay_path_length(_p(path), path.shape[0]))
