#!/usr/bin/env python
"""bench.py -- KKT factor+solves/sec on the BASELINE.json configurations.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config C4|C2|C1|C3] [--dump-outputs DIR]

One "step" (= one KKT unit) = one interior-point iteration's KKT work (SURVEY 8d): NT scaling of (v,s) ->
Atil = F^-T A -> H = Q + Atil'Atil (DMMA SYRK) -> [NCCL all-reduce of the partial Gram matrices when A is
row-sharded over N GPUs] -> Cholesky (+ Schur complement on G) -> k=2 solves (predictor + corrector
right-hand sides), each solve including its two A mat-vecs.  `value` times that with all inputs resident in
HBM; `e2e` times the same call sequence through the public API with HOST buffers (h2d of v,s and the
right-hand sides, d2h of lambda and the solutions inside the timed region).  The default workload is C4
(n=16384, m=262144: the configuration the metric is quoted on); the row shards make N>1 a strong-scaling
run of the same global problem.  Launch: one rank per GPU under torchrun (the driver's contract), or
`--gpus N` WITHOUT torchrun = ONE process driving N devices through a single handle (cip_options.ngpus).

`--impl reference` times the CPU restatement of the reference path (oracle/: NumPy + the BLAS/LAPACK routines
Julia's LinearAlgebra dispatches to -- dsyrk, dpotrf, dtrsv, dgemv) on the host cores.  Julia is not
installed in this image, so the reference itself cannot run (DESIGN.md).  The C4 unit is ~5 min of CPU work,
so the K timed steps together carry out ONE unit's work as far as a time budget allows: every step forms the
Gram contribution of a fresh slab of rows (+ its share of the four GEMVs), the last step runs the Cholesky
and the triangular solves at the real n.  Only the rows not reached are extrapolated (linearly, exact in
flops); `measured_fraction` says how much of the unit was measured.  `c2` is a second record where the
whole unit is measured on both arms.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "kkt_factor_plus_solves_per_sec"
UNIT = "kkt_units/s"
NSOLVES = 2
# name -> (n, m, description)
CONFIGS = {
    "C4": (16384, 262144, "dense QP n={n}, m={m} inequality rows, K=R^m, Q=diag+UU' (rank 32)"),
    "C2": (8192, 16384, "dense polyhedral QP n={n}, m={m} inequality rows, K=R^m, Q=diag+UU' (rank 32)"),
    "C1": (1000, 1000, "README nonnegative QP n={n}, Q=S'S (S~sprandn 0.1), A=I, K=R^n"),
    "C3": (4096, 16896, "SOCP n={n}, 512 Q-cones of dim 33 (m={m}) + equality block G (p=256)"),
    "C5": (20000, 22080, "MOI-shaped LP n={n}: x >= 0 plus one S block of order 64 (m={m}), sparse equality block G (p=1000), Q = 0"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C4", choices=list(CONFIGS))
    ap.add_argument("--n", type=int, default=0)
    ap.add_argument("--m", type=int, default=0)
    ap.add_argument("--no-solve", action="store_true", help="skip the full time-to-1e-8 solve")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-c2", action="store_true", help="skip the fully measured C2 sub-record")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity block")
    ap.add_argument("--cpu-budget", type=float, default=0.0,
                    help="seconds of CPU row work (default: 100 for --impl reference, 15 for the cpu_baseline leg)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed unit returned as DIR/<name>.npy (float64), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200 (the reference arm times synthetic row slabs, not a KKT unit)")
    return args


def workload_name(cfg, n, m):
    return f"{cfg}: " + CONFIGS[cfg][2].format(n=n, m=m) + f", k={NSOLVES} solves/unit"


# ------------------------------------------------------------------------------- CPU arm (oracle port)
def _cpu_threads():
    ncpu = str(os.cpu_count() or 1)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = ncpu           # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host thread
    try:
        import numpy  # noqa: F401  (loads OpenBLAS, so that the pool below exists and can be sized)
        import scipy.linalg  # noqa: F401
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=int(ncpu))
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return int(ncpu)


def cpu_unit_streamed(n, m, steps, warmup, budget_s):
    """One KKT unit of an R^m problem on the host cores with A streamed in row slabs (oracle.kkt.SlabbedCholKKT:
    dsyrk / dpotrf / dtrsv / dgemv, src/kktsolvers.jl:33-35,299,326-328).  The `steps` timed steps process
    distinct slabs covering a fraction f of the m rows (f = 1 if the budget allows); the last one also runs the
    Cholesky and the 2 x 2 triangular solves at the real n.  Returns a dict."""
    import numpy as np
    from oracle.kkt import SlabbedCholKKT
    rng = np.random.default_rng(0)
    K = SlabbedCholKKT(n, rng.uniform(1.0, 2.0, n))
    max_slab = max(256, min(8192, (1 << 30) // (8 * n) // 256 * 256))          # <= 1 GB of A per slab
    A_slab = rng.standard_normal((max_slab, n)) / math.sqrt(n)                # values do not matter for the timing
    dys = [rng.standard_normal(n) for _ in range(NSOLVES)]

    def row_step(rows, seed):
        """Gram contribution + the GEMV shares of NSOLVES solves for `rows` fresh rows; returns seconds."""
        r = np.random.default_rng(1000 + seed)
        t_total = 0.0
        done = 0
        while done < rows:
            k = min(max_slab, rows - done)
            f = r.uniform(0.5, 2.0, k)
            rv = r.standard_normal(k)
            A = A_slab[:k]
            t0 = time.perf_counter()
            K.add_rows(A, f)
            for s in range(NSOLVES):
                t1, _ = K.rhs_rows(A, f, rv)
                K.dv_rows(A, f, t1, dys[s])
            t_total += time.perf_counter() - t0
            done += k
        return t_total

    # calibration + warm-up (untimed): the BLAS thread pool and the page cache are warm afterwards
    cal_rows = min(m, 1024)
    t_cal = row_step(cal_rows, -1)
    for i in range(max(0, warmup - 1)):
        t_cal = min(t_cal, row_step(cal_rows, -2 - i))
    est_full = t_cal * m / cal_rows
    frac = min(1.0, budget_s / est_full)
    rows_step = max(256, int(frac * m / steps) // 256 * 256)
    rows_step = min(rows_step, max(256, m // steps // 256 * 256)) if m >= 256 * steps else max(1, m // steps)
    K.H[:] = 0.0
    step_s = []
    for i in range(steps):
        t = row_step(rows_step, i)
        if i == steps - 1:
            t0 = time.perf_counter()
            K.factor()
            t_chol = time.perf_counter() - t0
            t0 = time.perf_counter()
            for s in range(NSOLVES):
                K.solve(dys[s])
            t_trsv = time.perf_counter() - t0
            t += t_chol + t_trsv
        step_s.append(t)
    rows_meas = rows_step * steps
    t_rows = sum(step_s) - t_chol - t_trsv
    unit = t_rows * (m / rows_meas) + t_chol + t_trsv
    return {"unit_s": unit, "timed_s": sum(step_s), "step_s": step_s, "rows_measured": rows_meas,
            "rows_fraction": rows_meas / m, "time_fraction": sum(step_s) / unit, "t_rows_s": t_rows,
            "t_chol_s": t_chol, "t_trsv_s": t_trsv, "extrapolated": rows_meas < m}


def cpu_unit_oracle(prob, pts, rhs, repeats=1):
    """One KKT unit through the oracle's 3-level kktsolver protocol, fully measured (C1/C2/C3 sizes):
    LEVEL 2 = kktsolver_chol(Q,A,G,cone_dims)(F, F^-T), LEVEL 3 x NSOLVES.  Returns best seconds per unit."""
    import numpy as np
    import oracle as O
    gen = O.kktsolver_chol(prob["Q"], prob["A"], prob["G"], prob["cone_dims"])       # LEVEL 1 (untimed: upload)
    best = float("inf")
    for rep in range(repeats + 1):                                                   # first pass = warm-up
        v, s = pts[rep % len(pts)]
        t0 = time.perf_counter()
        blocks, off = [], 0
        for t, k in prob["cone_dims"]:                                               # nt_scaling, src/ConicIP.jl:589-605
            if t == "R":
                blocks.append(O.Diag(np.sqrt(s[off:off + k] / v[off:off + k])))
            elif t == "Q":
                blocks.append(O.nestod_soc(v[off:off + k], s[off:off + k]))
            else:
                blocks.append(O.nestod_sdc(v[off:off + k], s[off:off + k]))
            off += k
        F = O.Block(blocks)
        solve = gen(F, F.inv_adjoint())
        for ry, rw, rv in rhs:
            solve(ry, rw, rv)
        dt = time.perf_counter() - t0
        if rep > 0:
            best = min(best, dt)
    return best


def host_problem(cfg, n, m):
    """C1 / C3 (and C2 for the CPU sub-record) as NumPy problems + interior points and right-hand sides."""
    import numpy as np
    from conicip_b200 import problems as P
    if cfg == "C1":
        prob = P.config1(n=n)
    elif cfg == "C3":
        prob = P.config3(n=n, ncones=m // 33)
    elif cfg == "C5":
        prob = P.config5(n=n, k=64, p=1000 if n >= 20000 else max(8, n // 20))
    else:
        rng = np.random.default_rng(2)
        A = rng.standard_normal((m, n)) / math.sqrt(n)
        U = rng.standard_normal((n, 32)) / math.sqrt(32)
        prob = dict(name=cfg, Q=np.diag(rng.uniform(1.0, 2.0, n)) + U @ U.T, c=rng.standard_normal(n), A=A,
                    b=A @ rng.standard_normal(n) - rng.uniform(0.1, 1.1, m), cone_dims=[("R", m)],
                    G=np.zeros((0, n)), d=np.zeros(0))
    rng = np.random.default_rng(9)
    mm, p = prob["A"].shape[0], prob["G"].shape[0]

    def point():
        v, s = np.zeros(mm), np.zeros(mm)
        off = 0
        for t, k in prob["cone_dims"]:
            if t == "R":
                v[off:off + k] = rng.uniform(0.5, 1.5, k); s[off:off + k] = rng.uniform(0.5, 1.5, k)
            elif t == "Q":
                for x in (v, s):
                    u = rng.standard_normal(k - 1); x[off] = np.linalg.norm(u) + 0.5; x[off + 1:off + k] = u
            else:                                    # S: vecm of a well-conditioned positive definite matrix
                ks = int(round((math.sqrt(1 + 8 * k) - 1) / 2))
                for x in (v, s):
                    B = rng.standard_normal((ks, ks)) / math.sqrt(ks)
                    x[off:off + k] = P._svec(B @ B.T + 0.5 * np.eye(ks))
            off += k
        return v, s
    pts = [point(), point()]
    rhs = [(rng.standard_normal(len(prob["c"])), rng.standard_normal(p), rng.standard_normal(mm)) for _ in range(NSOLVES)]
    return prob, pts, rhs


def run_reference(args, n, m):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = _cpu_threads()
    steps, warmup = max(1, args.steps), args.warmup
    line = {"metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "reference", "config": {"workload": workload_name(args.config, n, m)}, "gpu_launches": 0}
    if args.config == "C4":
        budget = args.cpu_budget or 100.0
        r = cpu_unit_streamed(n, m, steps, warmup, budget)
        val = 1.0 / r["unit_s"]
        sample = (f"oracle port (oracle.kkt.SlabbedCholKKT: BLAS dsyrk Atil'Atil, LAPACK dpotrf, dtrsv, dgemv), "
                  f"{threads} threads; the {steps} timed steps together carry out one unit: Gram + GEMV shares of "
                  f"{r['rows_measured']} of {m} rows measured ({100 * r['rows_fraction']:.1f}%, {r['t_rows_s']:.1f} s), "
                  f"dpotrf at the real n={n} ({r['t_chol_s']:.1f} s) and {NSOLVES}x2 dtrsv ({r['t_trsv_s']:.2f} s) measured "
                  f"once; only the remaining rows are extrapolated (linear in m)")
        line.update({"value": val, "ms_per_step": 1e3 * r["timed_s"] / steps, "unit_ms": 1e3 * r["unit_s"],
                     "extrapolated": r["extrapolated"], "measured_fraction": r["rows_fraction"],
                     "measured_time_fraction": r["time_fraction"],
                     "ms_per_step_note": "wall time of one timed step (a bounded share of one unit); value = 1 / unit_ms"})
    else:
        prob, pts, rhs = host_problem(args.config, n, m)
        times = []
        for i in range(warmup + steps):
            t = cpu_unit_oracle(prob, pts, rhs, repeats=1)
            if i >= warmup:
                times.append(t)
        unit = sum(times) / len(times)
        val = 1.0 / unit
        sample = (f"oracle.kktsolver_chol through the 3-level protocol (LEVEL 2 + {NSOLVES} x LEVEL 3), {threads} threads, "
                  f"whole unit measured every step")
        line.update({"value": val, "ms_per_step": 1e3 * unit, "unit_ms": 1e3 * unit, "extrapolated": False,
                     "measured_fraction": 1.0})
    line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                            "extrapolated": line["extrapolated"], "measured_fraction": line["measured_fraction"]}
    line["e2e"] = {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if args.config == "C4" and not args.no_c2:
        n2, m2 = CONFIGS["C2"][0], CONFIGS["C2"][1]
        prob, pts, rhs = host_problem("C2", n2, m2)
        t = cpu_unit_oracle(prob, pts, rhs, repeats=1)
        line["c2"] = {"workload": workload_name("C2", n2, m2), "value": 1.0 / t, "unit": UNIT, "ms_per_unit": 1e3 * t,
                      "measured_fraction": 1.0, "extrapolated": False, "cores": threads,
                      "how": "oracle.kktsolver_chol, 3-level protocol, whole unit timed after one warm-up unit"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------- B200 arm
class Dist:
    """One rank per GPU under torchrun (world > 1), or a single process (world == 1)."""

    def __init__(self, torch):
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _red(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._red(x, self.dist.ReduceOp.MAX) if self.world > 1 else x

    def sum(self, x):
        return self._red(x, self.dist.ReduceOp.SUM) if self.world > 1 else x

    def min(self, x):
        return self._red(x, self.dist.ReduceOp.MIN) if self.world > 1 else x

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def device_qp(cb, torch, D, n, m, seed, ngpus_single=1):
    """C4 / C2: dense QP generated on the device (problems.config4_device), row-sharded over the ranks, or, for a
    single-process multi-GPU handle, generated whole on device 0 and sliced by the library (opts.ngpus)."""
    from conicip_b200 import problems as P
    from conicip_b200.dist import init_engine_comm
    prob = P.config4_device(n=n, m=m, seed=seed, rank=D.rank, nranks=D.world)
    eng = cb.Engine(prob["Q"], prob["At"].t(), None, prob["cone_dims"], ngpus=ngpus_single)
    out = dict(eng=eng, m_loc=prob["m_loc"], b=prob["b"], c=prob["c"], Q=prob["Q"], cone_dims=prob["cone_dims"])
    del prob["At"]
    torch.cuda.empty_cache()
    eng._bind_stream()
    if D.world > 1:
        init_engine_comm(eng)
    return out


def timed_unit_loop(torch, D, eng, pts, rhs, steps, warmup, sample_clocks):
    """W warm-up units, then exactly K timed units between barriers; CUDA events on the launching stream.
    Also returns what the last timed unit returned: lambda and one (dy, dw, dv) per right-hand side."""
    def unit(i):
        v, s = pts[i % len(pts)]
        lam = eng.factor_from_point(v, s)
        return lam, [eng.solve(ry, rw, rv) for ry, rw, rv in rhs]
    for i in range(warmup):
        unit(i)
    st0 = eng.stats()
    sampler = ClockSampler(D.local)
    if sample_clocks and D.rank == 0:
        sampler.start()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phases = {k: [] for k in ("ms_scale", "ms_syrk", "ms_allreduce", "ms_chol", "ms_schur", "ms_solve")}
    e0.record()
    for i in range(steps):
        last = unit(i)
        st = eng.stats()
        for k in phases:
            phases[k].append(st[k])
    e1.record()
    D.barrier()
    ms_total = D.max(e0.elapsed_time(e1))
    clocks = sampler.stop() if (sample_clocks and D.rank == 0) else None
    launches = eng.stats()["kernel_launches"] - st0["kernel_launches"]
    avg = {k: sum(v) / len(v) for k, v in phases.items()}
    return ms_total / steps, clocks, int(launches), avg, last


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(torch, D, out_dir, lam, sols):
    """Writes lambda and every solve's (dy, dw, dv) as out_dir/<name>.npy in float64.  m-length vectors of a torchrun
    launch are gathered to rank 0 first.  A vector longer than its share of DUMP_CAP_BYTES is replaced by the entries
    at a fixed seeded choice of indices, the same in every run of the same shape."""
    import numpy as np
    arrays = {"lambda": lam}
    for k, (dy, dw, dv) in enumerate(sols):
        arrays.update({f"dy{k}": dy, f"dw{k}": dw, f"dv{k}": dv})
    arrays = {k: x for k, x in arrays.items() if x is not None and len(x) > 0}
    if D.world > 1:                                   # lambda and dv are this rank's rows; dy is replicated
        arrays.update({k: _gather(torch, D, x) for k, x in arrays.items() if k == "lambda" or k.startswith("dv")})
    if D.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_CAP_BYTES // 8 // len(arrays)
    for k, x in arrays.items():
        x = x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)
        if x.size > share:
            x = x[np.sort(np.random.default_rng(0).choice(x.size, share, replace=False))]
        np.save(os.path.join(out_dir, f"{k}.npy"), x.astype(np.float64))
    print(f"[bench] wrote {', '.join(arrays)} to {out_dir}", file=sys.stderr, flush=True)


def e2e_unit_loop(torch, D, eng, pts, rhs, steps, n, m_loc, p):
    """The same unit through the public API with pinned HOST buffers (copies inside the timed region)."""
    pin = lambda t: None if t is None else t.cpu().pin_memory().numpy()
    h_pts = [(pin(v), pin(s)) for v, s in pts]
    h_rhs = [(pin(a), pin(b), pin(c)) for a, b, c in rhs]
    h2d = 8 * (2 * m_loc + len(rhs) * (n + p + m_loc))
    d2h = 8 * (m_loc + len(rhs) * (n + p + m_loc))

    def unit(i):
        v, s = h_pts[i % len(h_pts)]
        lam = eng.factor_from_point(v, s)
        return lam, [eng.solve(ry, rw, rv) for ry, rw, rv in h_rhs]
    unit(0)
    D.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        unit(i)
    D.barrier()
    ms = D.max((time.perf_counter() - t0) * 1e3) / steps
    return {"value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms,
            "h2d_bytes_per_step": int(D.sum(float(h2d))), "d2h_bytes_per_step": int(D.sum(float(d2h))),
            "timer": "host perf_counter around the API calls (each call blocks until outputs are on the host), max over ranks"}


def fp64_peaks(cb, torch):
    """FP64 ceilings measured in this run: cuBLAS DGEMM 8192^3 (the roofline denominator unless the driver's
    MEASURED_PEAKS.json carries an FP64 figure) and the register-only DMMA / DFMA loops of the library."""
    peaks = cb.measure_fp64_peaks()
    a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    b = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(3):
        a @ b
    g1.record()
    torch.cuda.synchronize()
    dgemm = 3 * 2 * 8192 ** 3 / (g0.elapsed_time(g1) * 1e-3) / 1e12
    driver = None
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        for k, v in mp.items():
            if ("fp64" in k.lower() or "f64" in k.lower()) and isinstance(v, (int, float)):
                driver = (k, float(v))
    except Exception:
        pass
    return peaks, dgemm, driver


def ncu_traffic(n, m_loc):
    """dram__bytes_read.sum + dram__bytes_write.sum of one SYRK launch at this shape from the committed
    `ncu --set full` captures (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep
    CSV export); null when no capture exists for the shape.  Not measurable inside an unprofiled run."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = tab.get(f"gemm_nt_syrk:n={n},m={m_loc}")
        return (e["dram_bytes"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


def run_b200(args, n, m):
    import numpy as np
    import torch

    import conicip_b200 as cb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the b200 arm)")
    D = Dist(torch)
    single_process = D.world == 1 and args.gpus > 1          # one process, one handle, N devices (opts.ngpus)
    ngpus_single = args.gpus if single_process else 1
    assert single_process or D.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={D.world}"
    rel = lambda a, b: float(torch.linalg.vector_norm(a - b) / torch.linalg.vector_norm(b))

    t_setup = time.time()
    cfg = args.config
    if cfg in ("C4", "C2"):
        assert m % (args.gpus * 32) == 0
        pr = device_qp(cb, torch, D, n, m, seed=4 if cfg == "C4" else 2, ngpus_single=ngpus_single)
        eng, m_loc, p = pr["eng"], pr["m_loc"], 0
        g = torch.Generator(device="cuda")
        g.manual_seed(100 + D.rank)
        rnd = lambda k, lo=0.0: torch.rand(k, generator=g, dtype=torch.float64, device="cuda") + lo
        pts = [(rnd(m_loc, 0.5), rnd(m_loc, 0.5)) for _ in range(2)]
        g.manual_seed(7)                                  # n-vectors are replicated across ranks
        rys = [torch.randn(n, generator=g, dtype=torch.float64, device="cuda") for _ in range(NSOLVES)]
        g.manual_seed(200 + D.rank)
        rhs = [(ry, None, torch.randn(m_loc, generator=g, dtype=torch.float64, device="cuda")) for ry in rys]
        c_vec, b_loc, d_vec = pr["c"], pr["b"], None
        hprob = None
    else:
        assert D.world == 1, "C1 / C3 / C5 are single-GPU bench lines"
        hprob, hpts, hrhs = host_problem(cfg, n, m)
        p = hprob["G"].shape[0]
        eng = cb.Engine(hprob["Q"], hprob["A"], hprob["G"] if p else None, hprob["cone_dims"], ngpus=ngpus_single)
        eng._bind_stream()
        T = lambda x: torch.as_tensor(x).cuda()
        pts = [(T(v), T(s)) for v, s in hpts]
        rhs = [(T(a), T(b) if p else None, T(c)) for a, b, c in hrhs]
        m_loc = hprob["A"].shape[0]
        c_vec, b_loc, d_vec = T(hprob["c"]), T(hprob["b"]), (T(hprob["d"]) if p else None)
    t_setup = time.time() - t_setup
    if D.rank == 0:
        print(f"[bench] setup {t_setup:.1f} s ({cfg}, n={n}, m={m}, gpus={args.gpus}, "
              f"{'single process' if single_process else 'torchrun' if D.world > 1 else 'one GPU'})", file=sys.stderr, flush=True)

    ms_step, clocks, launches, ph, (lam_last, sols_last) = timed_unit_loop(torch, D, eng, pts, rhs, args.steps, args.warmup, True)
    value = 1e3 / ms_step
    if D.rank == 0:
        print(f"[bench] device-resident: {ms_step:.2f} ms/step", file=sys.stderr, flush=True)
    if args.dump_outputs:
        dump_outputs(torch, D, args.dump_outputs, lam_last, sols_last)
    del lam_last, sols_last
    e2e = e2e_unit_loop(torch, D, eng, pts, rhs, max(2, min(args.steps, 3)), n, m_loc, p)

    # ---- roofline of the dominant kernel (gemm_nt as the SYRK), CUDA events recorded by the library on the
    #      launching stream around it inside the timed units
    syrk_flops = float(m // args.gpus) * n * n               # algorithmic m n^2 of one GPU's rows (SURVEY 8d)
    achieved = syrk_flops / (ph["ms_syrk"] * 1e-3) / 1e12
    peaks, dgemm_tf, driver_peak = fp64_peaks(cb, torch)
    peak = driver_peak[1] if driver_peak else dgemm_tf
    traffic, traffic_src = ncu_traffic(n, m_loc)
    roofline = {
        "bound": "tensor", "kernel": "gemm_nt_kernel (SYRK H = Q + Atil'Atil)", "achieved": achieved,
        "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": (f"MEASURED_PEAKS.json {driver_peak[0]}" if driver_peak else
                        "cuBLAS DGEMM 8192^3 FP64 measured in this run (MEASURED_PEAKS.json has no FP64 entry and the "
                        "profiling guide states no FP64 fallback)"),
        "cublas_dgemm_tflops": dgemm_tf, "dmma_register_peak_tflops": peaks["dmma_tflops"],
        "dfma_register_peak_tflops": peaks["dfma_tflops"], "frac_of_dmma_register_peak": achieved / peaks["dmma_tflops"],
        "flops_per_launch": syrk_flops, "ms_per_launch": ph["ms_syrk"],
        "step_breakdown_ms": {"scale_panel": ph["ms_scale"], "syrk": ph["ms_syrk"], "allreduce": ph["ms_allreduce"],
                              "cholesky": ph["ms_chol"], "schur": ph["ms_schur"], "solve_each": ph["ms_solve"]},
    }

    # ---- parity: the KKT unit just timed, checked inside this run
    parity = None
    if not args.no_parity:
        parity = {}
        v, s = pts[0]
        lam = eng.factor_from_point(v, s)
        ry, rw, rv = rhs[0]
        dy, dw, dv = eng.solve(ry, rw, rv)
        # (1) residual of the 3x3 system through the independent mat-vec kernels (R rows: F'F = diag(s/v))
        if cfg in ("C4", "C2"):
            r1 = eng.mul_Q(dy) - eng.mul_A(dv, trans=True) - ry
            r3 = eng.mul_A(dy) + (s / v) * dv - rv
            n3 = torch.linalg.vector_norm(r3) ** 2
            d3 = torch.linalg.vector_norm(rv) ** 2
            parity["kkt_unit_residual"] = {
                "row1_rel": float(torch.linalg.vector_norm(r1) / torch.linalg.vector_norm(ry)),
                "row3_rel": math.sqrt(D.sum(float(n3)) / D.sum(float(d3)))}
        parity["dy_norm"] = float(torch.linalg.vector_norm(dy))
        # (2) N > 1: the sharded unit against the SAME unit on one GPU (rank 0 builds the whole problem)
        if args.gpus > 1 and cfg in ("C4", "C2"):
            free, _ = torch.cuda.mem_get_info()
            need = 2.2 * 8.0 * n * m + 5 * 8.0 * n * n
            if free > need + 4e9:
                gather = (lambda x: _gather(torch, D, x)) if D.world > 1 else (lambda x: x)
                v_all, s_all, rv_all, lam_all, dv_all = gather(v), gather(s), gather(rv), gather(lam), gather(dv)
                if D.rank == 0:
                    from conicip_b200 import problems as P
                    full = P.config4_device(n=n, m=m, seed=4 if cfg == "C4" else 2, rank=0, nranks=1)
                    e1 = cb.Engine(full["Q"], full["At"].t(), None, full["cone_dims"])
                    del full["At"]
                    torch.cuda.empty_cache()
                    e1._bind_stream()
                    lam1 = e1.factor_from_point(v_all, s_all)
                    dy1, _, dv1 = e1.solve(ry, None, rv_all)
                    parity["vs_single_gpu"] = {"rel_lambda": rel(lam_all, lam1), "rel_dy": rel(dy, dy1),
                                               "rel_dv": rel(dv_all, dv1), "dy_norm_single": float(torch.linalg.vector_norm(dy1))}
                    e1.close()
                    del e1
                    torch.cuda.empty_cache()
                D.barrier()
            else:
                parity["vs_single_gpu"] = f"skipped: {free / 1e9:.0f} GB free on rank 0, {need / 1e9:.0f} GB needed"
            # (3) block-cyclic distributed Cholesky against the replicated single-GPU factorisation of the same H
            os.environ["CIP_DIST_CHOL"] = "0"
            eng.factor_from_point(v, s)
            dy_r, _, dv_r = eng.solve(ry, rw, rv)
            os.environ["CIP_DIST_CHOL"] = "1"
            eng.factor_from_point(v, s)
            dy_d, _, dv_d = eng.solve(ry, rw, rv)
            os.environ.pop("CIP_DIST_CHOL")
            parity["dist_vs_replicated_cholesky"] = {"dy_bit_identical": bool(torch.equal(dy_r, dy_d)),
                                                     "rel_dy": rel(dy_d, dy_r)}

    # ---- full interior-point solve: time-to-1e-8 (native loop: one cip_ipm_solve call per rank)
    solve_info = None
    if not args.no_solve:
        # small configurations: the first call also pays one-time costs (lazy loading of the kernels only the loop uses,
        # pool allocation), which vary from box to box and dwarf a 10 ms solve -- time a second call and report both
        t_calls = []
        for _ in range(1 if cfg == "C4" else 2):
            D.barrier()
            t0 = time.perf_counter()
            y, w, vv, info = eng.ipm_solve(c_vec, b_loc, d_vec, optTol=1e-8)
            D.barrier()
            t_calls.append(D.max(time.perf_counter() - t0))
        t_solve = min(t_calls)
        solve_info = {"time_to_1e-8_s": t_solve, "first_call_s": t_calls[0], "status": info["status"], "iterations": info["Iter"],
                      "factors": info["factors"], "solves": info["solves"], "prFeas": info["prFeas"],
                      "duFeas": info["duFeas"], "muFeas": info["muFeas"], "pobj": info["pobj"], "dobj": info["dobj"],
                      "driver": "cip_ipm_solve (native)"}
        if hprob is not None and D.world == 1 and ngpus_single == 1:
            # the host-driven path beside the native loop: conicip_b200.conicIP is the reference's loop structure
            # (src/ConicIP.jl:468-939) on the host, calling LEVEL 1 / 2 / 3 and every cone kernel through the C ABI one
            # call at a time -- what a host driver that keeps `conicIP` pays; the time includes LEVEL 1 (the upload)
            t_host = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                hs = cb.conicIP(hprob["Q"], hprob["c"], hprob["A"], hprob["b"], hprob["cone_dims"],
                                hprob["G"] if p else None, hprob["d"] if p else None, optTol=1e-8)
                t_host.append(time.perf_counter() - t0)
            solve_info["host_driver"] = {"time_to_1e-8_s": min(t_host), "first_call_s": t_host[0], "status": hs.status,
                                         "iterations": hs.Iter, "factors": hs.factors, "solves": hs.solves,
                                         "driver": "conicip_b200.conicIP (host loop, one C-ABI call per kktsolver level and cone kernel; includes cip_create)"}
        if parity is not None:
            # the solution itself, to compare across the N = 1, 2, 4, 8 lines, and an independent evaluation of the
            # optimality conditions of  min 1/2 y'Qy - c'y  s.t. Ay - b in K  through the mat-vec kernels
            probe = torch.cos(torch.arange(n, dtype=torch.float64, device="cuda"))
            fs = {"y_norm": float(torch.linalg.vector_norm(y)), "y_probe": float(torch.dot(y, probe))}
            if cfg in ("C4", "C2"):
                slack = eng.mul_A(y) - b_loc
                stat = eng.mul_Q(y) - c_vec - eng.mul_A(vv, trans=True)
                fs["stationarity_rel"] = float(torch.linalg.vector_norm(stat) / (1 + torch.linalg.vector_norm(c_vec)))
                fs["min_slack"] = D.min(float(slack.min()))
                fs["min_v"] = D.min(float(vv.min()))
                fs["complementarity"] = abs(D.sum(float(torch.dot(slack, vv)))) / m
            parity["full_solve"] = fs

    # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    if D.rank == 0 and args.gpus == 1 and not args.no_cpu:
        threads = _cpu_threads()
        if cfg in ("C4", "C2"):
            r = cpu_unit_streamed(n, m, 4, 2, args.cpu_budget or 15.0)
            cpu = {"value": 1.0 / r["unit_s"], "unit": UNIT, "cores": threads, "kind": "port",
                   "extrapolated": r["extrapolated"], "measured_fraction": r["rows_fraction"],
                   "sample": (f"oracle.kkt.SlabbedCholKKT (dsyrk / dpotrf / dtrsv / dgemv), {threads} threads: Gram + GEMV "
                              f"shares of {r['rows_measured']} of {m} rows ({r['t_rows_s']:.1f} s, rest linear in m), dpotrf "
                              f"at the real n={n} ({r['t_chol_s']:.1f} s), {NSOLVES}x2 dtrsv ({r['t_trsv_s']:.2f} s); "
                              f"`bench.py --impl reference` measures a larger share")}
        else:
            reps = 1 if cfg == "C5" else 2           # a C5 unit is ~a minute of host time: one warm-up + one timed pass
            t = cpu_unit_oracle(hprob, hpts, hrhs, repeats=reps)
            cpu = {"value": 1.0 / t, "unit": UNIT, "cores": threads, "kind": "port", "extrapolated": False,
                   "measured_fraction": 1.0,
                   "sample": f"oracle.kktsolver_chol through the 3-level protocol, whole unit, best of {reps}, {threads} threads"}

    # ---- C2: a second record where the whole unit is measured on both arms (N = 1, default workload only)
    c2 = None
    if cfg == "C4" and args.gpus == 1 and not args.no_c2:
        eng.close()
        del eng, pts, rhs
        torch.cuda.empty_cache()
        n2, m2 = CONFIGS["C2"][0], CONFIGS["C2"][1]
        pr2 = device_qp(cb, torch, D, n2, m2, seed=2)
        g = torch.Generator(device="cuda"); g.manual_seed(300)
        rnd = lambda k, lo=0.0: torch.rand(k, generator=g, dtype=torch.float64, device="cuda") + lo
        pts2 = [(rnd(m2, 0.5), rnd(m2, 0.5)) for _ in range(2)]
        rhs2 = [(torch.randn(n2, generator=g, dtype=torch.float64, device="cuda"), None,
                 torch.randn(m2, generator=g, dtype=torch.float64, device="cuda")) for _ in range(NSOLVES)]
        ms2, _, l2, ph2, _ = timed_unit_loop(torch, D, pr2["eng"], pts2, rhs2, max(args.steps, 10), max(args.warmup, 3), False)
        e2e2 = e2e_unit_loop(torch, D, pr2["eng"], pts2, rhs2, 5, n2, m2, 0)
        c2 = {"workload": workload_name("C2", n2, m2), "value": 1e3 / ms2, "unit": UNIT, "ms_per_step": ms2,
              "e2e": {k: e2e2[k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step")},
              "gpu_launches_per_step": l2 / max(args.steps, 10),
              "syrk_tflops": float(m2) * n2 * n2 / (ph2["ms_syrk"] * 1e-3) / 1e12,
              "cholesky_tflops": float(n2) ** 3 / 3 / (ph2["ms_chol"] * 1e-3) / 1e12,
              "step_breakdown_ms": {"scale_panel": ph2["ms_scale"], "syrk": ph2["ms_syrk"], "cholesky": ph2["ms_chol"],
                                    "solve_each": ph2["ms_solve"]},
              "cpu_reference": "the `c2` record of `bench.py --impl reference` is the fully measured CPU unit of this shape"}
        pr2["eng"].close()

    if D.rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(cfg, n, m), "rows_per_gpu": m // args.gpus,
                       "l2": "inputs larger than L2 (A slab %.2f GB per GPU re-read every step)" % (m / args.gpus * n * 8 / 1e9),
                       "launch": ("single process, one handle, cip_options.ngpus" if single_process else
                                  "one process per GPU (torchrun)" if D.world > 1 else "single GPU"),
                       "setup_s": t_setup},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "parity": parity, "full_solve": solve_info, "c2": c2,
        }
        print(json.dumps(line), flush=True)
    D.close()


def _gather(torch, D, x):
    """all-gather equal-length shard vectors to every rank (rank order = row order)."""
    out = [torch.empty_like(x) for _ in range(D.world)]
    D.dist.all_gather(out, x.contiguous())
    return torch.cat(out)


def main():
    args = parse()
    n, m = CONFIGS[args.config][0], CONFIGS[args.config][1]
    n, m = args.n or n, args.m or m
    if args.impl == "reference":
        run_reference(args, n, m)
    else:
        run_b200(args, n, m)


if __name__ == "__main__":
    main()
