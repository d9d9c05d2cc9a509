"""Folded R + Q SYRK (fold_scaling = 1 with Q cones) against the materialised one (fold_scaling = 2).

1. C3 shape (n = 4096, 512 cones of dimension 33, p = 256): SYRK time (cip_stats.ms_syrk) and scaling pass time
   (ms_scale: Atil = F^-T A when materialised, the T pass when folded), the two handles alternating, --runs each;
   device_bytes of both; max |H_fold - H_mat| relative to max |H|.
2. A large SOCP (n = 16384, cones of dimension 33, m chosen so that A fills --frac of device memory): the
   materialised handle must fail to create, the folded one solves to 1e-8 (time and iterations).

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


def c3_syrk(out, runs, gpu):
    import conicip_b200 as cb
    from conicip_b200 import problems as P
    prob = P.config3()
    G = prob["G"]
    cd = prob["cone_dims"]
    eng = {"materialised": cb.Engine(prob["Q"], prob["A"], G, cd, fold_scaling=2),
           "folded": cb.Engine(prob["Q"], prob["A"], G, cd, fold_scaling=1)}
    rng = np.random.default_rng(0)
    v, s = interior(cd, rng), interior(cd, rng)
    for e in eng.values():                      # warm-up: module load, tensor maps, first launches
        e.factor_from_point(v, s)
    times = {k: {"syrk": [], "scale": []} for k in eng}
    for _ in range(runs):                       # the two handles alternate; cip_stats holds the events of the last factor
        for k, e in eng.items():
            e.factor_from_point(v, s)
            st = e.stats()
            times[k]["syrk"].append(st["ms_syrk"])
            times[k]["scale"].append(st["ms_scale"])
    H = {}
    for k, e in eng.items():                    # H itself (before the Cholesky overwrites it)
        e.nt_scaling(v, s)
        e.form_H()
        H[k] = e.get_H()
    diff = float(np.max(np.abs(np.tril(H["folded"] - H["materialised"]))) / np.max(np.abs(H["materialised"])))
    rec = dict(what="C3_syrk", gpu=gpu, n=prob["A"].shape[1], m=prob["A"].shape[0], p=G.shape[0], runs=runs,
               bitwise_equal_H=bool(np.array_equal(H["folded"].view(np.uint64), H["materialised"].view(np.uint64))),
               max_rel_diff_H=diff)
    for k in eng:
        rec[f"{k}_ms_syrk"] = times[k]["syrk"]
        rec[f"{k}_ms_scale"] = times[k]["scale"]
        rec[f"{k}_ms_syrk_median"] = float(np.median(times[k]["syrk"]))
        rec[f"{k}_ms_scale_median"] = float(np.median(times[k]["scale"]))
        rec[f"{k}_device_bytes"] = eng[k].stats()["device_bytes"]
    rec["syrk_cost_pct"] = 100.0 * (rec["folded_ms_syrk_median"] / rec["materialised_ms_syrk_median"] - 1.0)
    emit(out, rec)
    for e in eng.values():
        e.close()


def large_socp(out, frac, n, k, gpu, optTol, verbose=False):
    import torch
    import conicip_b200 as cb
    from conicip_b200 import _lib
    total = torch.cuda.get_device_properties(0).total_memory
    ncones = int(frac * total / (8 * n) // k)
    m = ncones * k
    need = m * n * 8
    avail = 0
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    if avail < 1.15 * need:
        emit(out, dict(what="large_socp", gpu=gpu, error=f"host memory {avail / 1e9:.0f} GB < A {need / 1e9:.0f} GB"))
        return
    t0 = time.time()
    # A (m x n) column-major on the host = At (n x m) row-major, filled from the device in column blocks
    At = np.empty((n, m))
    g = torch.Generator(device="cuda")
    g.manual_seed(17)
    for j0 in range(0, n, 256):
        j1 = min(n, j0 + 256)
        At[j0:j1] = (torch.randn((j1 - j0, m), generator=g, dtype=torch.float64, device="cuda") / n ** 0.5).cpu().numpy()
    A = At.T                                   # Fortran-ordered view, no copy
    rng = np.random.default_rng(18)
    cd = [("Q", k)] * ncones
    y0 = rng.standard_normal(n)
    b = A @ y0 - interior(cd, rng)
    c = rng.standard_normal(n)
    Q = np.eye(n)
    t_gen = time.time() - t0
    rec = dict(what="large_socp", gpu=gpu, n=n, m=m, cone_dim=k, ncones=ncones, A_bytes=need,
               A_frac_of_device=need / total, host_gen_s=t_gen)
    for mode, name in ((2, "materialised"), (1, "folded")):
        torch.cuda.empty_cache()
        t0 = time.time()
        try:
            e = cb.Engine(Q, A, None, cd, fold_scaling=mode)
        except Exception as ex:                # expected for the materialised handle: the second copy does not fit
            rec[f"{name}_create"] = f"failed: {ex}"
            continue
        rec[f"{name}_create_s"] = time.time() - t0
        rec[f"{name}_device_bytes"] = e.stats()["device_bytes"]
        t0 = time.time()
        y, w, v, info = e.ipm_solve(c, b, None, optTol=optTol, verbose=verbose)
        st = e.stats()
        rec[name] = dict(solve_s=time.time() - t0, status=info["status"], iters=info["Iter"], factors=info["factors"],
                         prFeas=info["prFeas"], duFeas=info["duFeas"], muFeas=info["muFeas"],
                         last_ms_syrk=st["ms_syrk"], last_ms_scale=st["ms_scale"], last_ms_chol=st["ms_chol"],
                         last_error=_lib.last_error() if info["status"] == "Error" else "")
        e.close()
    rec["optTol"] = optTol
    emit(out, rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--frac", type=float, default=0.6)
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--k", type=int, default=33)
    ap.add_argument("--skip-large", action="store_true")
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--verbose", action="store_true", help="per-iteration residuals of the large solves")
    ap.add_argument("--out", default="fold_q_timing.jsonl")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fold_q_timing.py needs a CUDA (sm_100a) device")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    gpu = gpu_info()
    with open(a.out, "w") as out:
        if not a.skip_c3:
            c3_syrk(out, a.runs, gpu)
        if not a.skip_large:
            large_socp(out, a.frac, a.n, a.k, gpu, 1e-8, a.verbose)


if __name__ == "__main__":
    main()
