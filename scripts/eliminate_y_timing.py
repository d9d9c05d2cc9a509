"""The m-space form (eliminate_y = 1) against the n-space form (eliminate_y = 2) on wide problems with Q = I.

1. n = --n (16384), m in --ms (1024 .. 8192), R + Q cones (half the rows in R cones, half in Q cones of dimension
   64), p = --p equality rows, dense A.  Both handles alternate in one process: the time of one KKT unit
   (factor_from_point + 2 solves, synchronised wall clock, median of --runs), the phases of cip_stats, the time to 1e-8
   (cip_ipm_solve) and iterations, the resident bytes, and the create-time SYRK C = A D^-1 A' (CUDA kernel time of
   the gemm_nt launches inside cip_create, torch.profiler).
2. --reach: n = 150 000, m = 2 048, p = 64, A generated on the device, default options (auto must choose the
   m-space form): create time, resident bytes, iterations and time to 1e-8.

Writes one JSON line per measurement to stdout and to --out.  Needs a B200 (sm_100a).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def interior(cone_dims, rng):
    x = []
    for t, k in cone_dims:
        if t == "R":
            x.append(rng.uniform(0.5, 1.5, k))
        else:
            u = 0.2 * rng.standard_normal(k - 1)
            x.append(np.concatenate([[1.0 + np.linalg.norm(u)], u]))
    return np.concatenate(x)


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()


def cones_for(m):
    nq = (m // 2) // 64
    return [("R", m - 64 * nq)] + [("Q", 64)] * nq


def problem(n, m, p, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    At = torch.randn((n, m), generator=g, device="cuda", dtype=torch.float64) / np.sqrt(n)
    Gt = torch.randn((n, p), generator=g, device="cuda", dtype=torch.float64) / np.sqrt(n)
    cones = cones_for(m)
    y0 = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    s0 = torch.tensor(interior(cones, np.random.default_rng(seed)), device="cuda")
    A, G = At.t(), Gt.t()
    c = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    return dict(A=A, G=G, b=A @ y0 - s0, d=G @ y0, c=c, cones=cones)


def create(pr, n, ey):
    import scipy.sparse as sp
    import torch
    import conicip_b200 as cb
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e = cb.Engine(sp.identity(n, format="csr"), pr["A"], pr["G"], pr["cones"], eliminate_y=ey)
    e.sync()
    return e, time.perf_counter() - t0


def syrk_at_create(pr, n):
    """CUDA time of the gemm_nt launches (C, E', P and their split-K reductions) inside cip_create, m-space form."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e, _ = create(pr, n, 1)
        torch.cuda.synchronize()
    us = sum(ev.device_time_total for ev in prof.key_averages()
             if "gemm_nt" in ev.key or "splitk_reduce" in ev.key)
    e.close()
    return us / 1000.0


def unit_ms(e, pr, v, s, runs):
    import torch
    n, m, p = e.n, e.m, e.p
    rng = np.random.default_rng(1)
    T = lambda x: torch.tensor(x, device="cuda")
    ry, rw, rv = T(rng.standard_normal(n)), T(rng.standard_normal(p)), T(rng.standard_normal(m))
    vt, st = T(v), T(s)
    e.factor_from_point(vt, st)          # warm-up (graphs captured, modules loaded)
    e.solve(ry, rw, rv)
    ts, phases = [], []
    for _ in range(runs):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e.factor_from_point(vt, st)
        e.solve(ry, rw, rv)
        e.solve(ry, rw, rv)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
        so = e.stats()
        phases.append({k: so[k] for k in ("ms_scale", "ms_syrk", "ms_chol", "ms_schur", "ms_solve")})
    i = int(np.argsort(ts)[len(ts) // 2])
    return float(np.median(ts)), phases[i], [float(x) for x in ts]


def sweep(out, args, gpu):
    n, p = args.n, args.p
    for m in args.ms:
        pr = problem(n, m, p, seed=m)
        rec = dict(what="unit", n=n, m=m, p=p, gpu=gpu)
        rec["create_syrk_ms_m_space"] = syrk_at_create(pr, n)
        eng = {}
        for ey in (1, 2):
            e, tc = create(pr, n, ey)
            assert e.kkt_form_info()["eliminate_y"] == (1 if ey == 1 else 0)
            eng[ey] = e
            rec[f"create_s_{'m' if ey == 1 else 'n'}"] = tc
            rec[f"device_bytes_{'m' if ey == 1 else 'n'}"] = e.stats()["device_bytes"]
        rng = np.random.default_rng(2)
        v, s = interior(pr["cones"], rng), interior(pr["cones"], rng)
        res = {1: [], 2: []}
        for r in range(2):                   # alternate the two forms
            for ey in ((1, 2) if r == 0 else (2, 1)):
                res[ey].append(unit_ms(eng[ey], pr, v, s, args.runs))
        for ey, tag in ((1, "m"), (2, "n")):
            allt = sorted(t for x in res[ey] for t in x[2])
            rec[f"unit_ms_{tag}"] = float(np.median(allt))
            rec[f"unit_ms_{tag}_spread"] = [allt[0], allt[-1]]
            rec[f"phases_{tag}"] = res[ey][-1][1]
        # time to 1e-8, alternating
        for ey, tag in ((1, "m"), (2, "n")):
            y, w, vv, info = eng[ey].ipm_solve(pr["c"], pr["b"], pr["d"], optTol=1e-8)
            rec[f"ipm_{tag}"] = dict(status=info["status"], Iter=info["Iter"], seconds=info["seconds"],
                                     factors=info["factors"], solves=info["solves"])
            if ey == 1:
                y1 = y.clone()
            else:
                rec["rel_y_m_vs_n"] = float((y1 - y).norm() / y.norm())
        for e in eng.values():
            e.close()
        emit(out, rec)
        del pr
        import torch
        torch.cuda.empty_cache()


def reach(out, gpu):
    import torch
    n, m, p = 150_000, 2048, 64
    pr = problem(n, m, p, seed=7)
    e, tc = create(pr, n, 0)
    fi = e.kkt_form_info()
    y, w, v, info = e.ipm_solve(pr["c"], pr["b"], pr["d"], optTol=1e-8)
    torch.cuda.synchronize()
    rdu = float((y + pr["G"].t() @ w - pr["A"].t() @ v - pr["c"]).norm()) / (1 + float(pr["c"].norm()))
    emit(out, dict(what="reach", n=n, m=m, p=p, gpu=gpu, form=fi, create_s=tc,
                   device_bytes=e.stats()["device_bytes"], n_space_bytes_from_shapes=2 * ((n + 127) // 128 * 128) ** 2 * 8,
                   status=info["status"], Iter=info["Iter"], seconds=info["seconds"], dual_residual=rdu,
                   prFeas=info["prFeas"], duFeas=info["duFeas"], muFeas=info["muFeas"]))
    e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--ms", type=int, nargs="*", default=[1024, 2048, 4096, 8192])
    ap.add_argument("--p", type=int, default=64)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reach", action="store_true")
    ap.add_argument("--out", default="eliminate_y_timing.jsonl")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eliminate_y_timing needs a CUDA (sm_100a) device")
    gpu = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        if args.ms:
            sweep(out, args, gpu)
        if args.reach:
            reach(out, gpu)


if __name__ == "__main__":
    main()
