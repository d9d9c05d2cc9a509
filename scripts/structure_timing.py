"""cip_options.row_structure modes side by side, alternating in one process: KKT unit time and its phases, resident
bytes, time to 1e-8 through cip_ipm_solve, and how far the modes' results are apart.

    python scripts/structure_timing.py --out DIR [--units 5] [--warmup 2] [--only C5,C1,...] [--modes 0,1]

Workloads: C5 at full size through dense input and through a CSC copy of A, C1, a box QP (A = [I; -I], dense Q),
and a dense R-only QP with n bound rows appended (C2 plus I: the rest stays full width).  With mode 2 among the
modes (or when named in --only) also C5_rho0 (C5 with aug_rho = 0, so G couples no column) and C5_wide
(config5_sparse at n = 150 000, CSC input, no Q, aug_rho = 0).  C5_wide runs in mode 2 only: modes 0 and 1 hold
n_pad^2 doubles per H and Q, which the record computes from the shape instead of attempting.  A unit is what
bench.py times: factor at an interior point (NT scaling, H, Cholesky, Schur complement) plus two solves.  Writes
one JSON file per workload into DIR: r03_structure_<name>.json for the default modes 0,1 (keys "off" / "on"),
r04_split_<name>.json otherwise (keys "mode<k>")."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402

import conicip_b200 as cb  # noqa: E402
from conicip_b200 import problems as P  # noqa: E402

PHASES = ("ms_scale", "ms_syrk", "ms_chol", "ms_schur", "ms_solve")


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)) if b.size else 0.0


def interior(cone_dims, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(2):
        x = []
        for t, k in cone_dims:
            if t == "R":
                x.append(rng.uniform(0.5, 1.5, k))
            elif t == "Q":
                u = 0.2 * rng.standard_normal(k - 1)
                x.append(np.concatenate([[1.0 + np.linalg.norm(u)], u]))
            else:
                o = int(round((np.sqrt(1 + 8 * k) - 1) / 2))
                B = rng.standard_normal((o, o)) / np.sqrt(o)
                x.append(P._svec(B @ B.T + np.eye(o)))
        out.append(np.concatenate(x))
    return out


def workloads(only, modes):
    def c5():
        return P.config5()

    def c5_csc():
        p = P.config5()
        p["A_input"] = sp.csc_matrix(p["A"])
        return p

    def box():
        n = 8192
        rng = np.random.default_rng(8)
        p = P.box_qp(n)
        p["Q"] = P._lowrank_q(rng, n)
        p["name"] = "box_qp_8192"
        return p

    def c2_bounds():
        base = P.config2()
        n = base["A"].shape[1]
        rng = np.random.default_rng(9)
        A = np.vstack([base["A"], np.eye(n)])
        y0 = rng.uniform(0.5, 1.5, n)
        s0 = rng.uniform(0.1, 1.1, A.shape[0])
        return P._prob("C2_plus_bounds", base["Q"], base["c"], A, A @ y0 - s0, [("R", A.shape[0])], optTol=1e-8)

    def c5_rho0():
        p = P.config5()
        p["engine_kw"] = dict(aug_rho=0.0)
        return p

    def c5_wide():
        p = P.config5_sparse(n=150_000)
        p["A_input"], p["Q"] = p["A"], None
        p["engine_kw"] = dict(aug_rho=0.0)
        p["modes"] = (2,)
        return p

    table = {"C5": c5, "C5_csc": c5_csc, "C1": lambda: P.config1(), "box_qp": box, "C2_bounds": c2_bounds}
    split_table = {"C5_rho0": c5_rho0, "C5_wide": c5_wide}
    if 2 in modes or any(k in split_table for k in only):
        table.update(split_table)
    return [(k, f) for k, f in table.items() if not only or k in only]


def unit(e, v, s, ry, rw, rv):
    t0 = time.perf_counter()
    lam = e.factor_from_point(v, s)
    st = e.stats()
    ph = {k: st[k] for k in PHASES[:-1]}
    d1 = e.solve(ry, rw, rv)
    d2 = e.solve(0.5 * ry, rw, 2.0 * rv)
    ph["ms_solve"] = e.stats()["ms_solve"]
    return (time.perf_counter() - t0) * 1e3, ph, lam, d1, d2


def run(name, make, units, warmup, out_dir, gpu, modes):
    prob = make()
    A = prob.get("A_input", prob["A"])
    G = prob["G"] if prob["G"].shape[0] else None
    kw = prob.get("engine_kw", {})
    # a workload that names its modes (C5_wide: 2 only) is too large for the others, whatever --modes asks for
    skipped = [m for m in (0, 1, 2) if m not in prob["modes"]] if "modes" in prob else []
    modes = tuple(m for m in modes if m in prob.get("modes", modes))
    legacy = modes == (0, 1)
    label = {0: "off", 1: "on"} if legacy else {m: f"mode{m}" for m in modes}
    t0 = time.perf_counter()
    eng = {}
    setup = {}
    for mode in modes:
        t = time.perf_counter()
        eng[mode] = cb.Engine(prob["Q"], A, G, prob["cone_dims"], row_structure=mode, **kw)
        setup[mode] = time.perf_counter() - t
    gen_s = time.perf_counter() - t0
    e1 = eng[modes[-1]]
    v, s = interior(prob["cone_dims"], 1)
    rng = np.random.default_rng(2)
    ry, rw, rv = rng.standard_normal(e1.n), rng.standard_normal(e1.p) if e1.p else None, rng.standard_normal(e1.m)
    res = {m: {"unit_ms": [], "phases": []} for m in modes}
    outs = {}
    for it in range(warmup + units):
        for mode in modes:                        # alternate the modes
            ms, ph, lam, d1, d2 = unit(eng[mode], v, s, ry, rw, rv)
            outs[mode] = (lam, d1, d2)
            if it >= warmup:
                res[mode]["unit_ms"].append(ms)
                res[mode]["phases"].append(ph)
    summary = {}
    for mode in modes:
        r = res[mode]
        st = eng[mode].stats()
        summary[mode] = {
            "unit_ms_median": float(np.median(r["unit_ms"])), "unit_ms": r["unit_ms"],
            "phases_ms_median": {k: float(np.median([p[k] for p in r["phases"]])) for k in PHASES},
            "syrk_flops": st["syrk_flops"], "device_bytes": int(st["device_bytes"]), "create_s": setup[mode],
            "structure": eng[mode].structure_info(),
        }
        if mode == 2:
            summary[mode]["split"] = eng[mode].split_info()
    lo, hi = modes[0], modes[-1]
    lam0, a0, b0 = outs[lo]
    lam1, a1, b1 = outs[hi]
    diffs = {"lambda": rel(lam1, lam0), "dy": max(rel(a1[0], a0[0]), rel(b1[0], b0[0])),
             "dv": max(rel(a1[2], a0[2]), rel(b1[2], b0[2])),
             "dw": max(rel(a1[1], a0[1]), rel(b1[1], b0[1])) if e1.p else 0.0}
    full = {}
    sols = {}
    for mode in modes:
        t = time.perf_counter()
        y, w, vv, info = eng[mode].ipm_solve(prob["c"], prob["b"], prob["d"] if e1.p else None, optTol=1e-8)
        full[mode] = {"wall_s": time.perf_counter() - t, "seconds": info["seconds"], "status": info["status"],
                      "iterations": info["Iter"], "factors": info["factors"], "solves": info["solves"]}
        sols[mode] = (y, w, vv)
    diffs.update({"full_y": rel(sols[hi][0], sols[lo][0]), "full_v": rel(sols[hi][2], sols[lo][2]),
                  "full_w": rel(sols[hi][1], sols[lo][1]) if e1.p else 0.0})
    for e in eng.values():
        e.close()
    rec = {"workload": name, "n": e1.n, "m": e1.m, "p": e1.p, "input": "csc" if "A_input" in prob else "dense",
           "gpu": gpu, "units": units, "warmup": warmup, "setup_s": gen_s}
    if kw:
        rec["engine_options"] = kw
    for mode in modes:
        rec[label[mode]] = {**summary[mode], "full_solve": full[mode]}
    if len(modes) > 1:
        rec["max_rel_diff_on_vs_off" if legacy else f"max_rel_diff_mode{hi}_vs_mode{lo}"] = diffs
    if skipped:
        n_pad = -(-e1.n // 128) * 128
        rec["not_attempted"] = {f"mode{m}": f"computed from the shape, not run: needs n_pad^2 doubles for H and for Q, "
                                            f"2 x {8 * n_pad * n_pad / 1e9:.0f} GB (n_pad = {n_pad}), more than the "
                                            f"device holds" for m in skipped}
    rec["timer"] = ("unit: host perf_counter around factor_from_point + 2 solves (host outputs: each call syncs); "
                    "phases: CUDA events of cip_stats; full solve: cip_ipm_result.seconds")
    print(json.dumps(rec), flush=True)
    if out_dir:
        fname = f"r03_structure_{name}.json" if legacy else f"r04_split_{name}.json"
        with open(os.path.join(out_dir, fname), "w") as f:
            json.dump(rec, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--units", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="")
    ap.add_argument("--modes", default="0,1", help="row_structure modes to compare, e.g. 1,2")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("structure_timing.py needs the GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    gpu = q[0] if q else "unknown"
    print("gpu:", gpu, flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    only = [s for s in a.only.split(",") if s]
    modes = tuple(sorted({int(x) for x in a.modes.split(",") if x}))
    for name, make in workloads(only, modes):
        run(name, make, a.units, a.warmup, a.out, gpu, modes)


if __name__ == "__main__":
    main()
