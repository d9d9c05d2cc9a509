"""Phase timing of the fast SYRK of form_H (csrc/fast_syrk.cu) against the classical SYRK, on the device-generated
dense QP of bench.py (problems.config4_device, all rows R).

For each shape (default n in {8192, 12288, 16384} with m = 16 n, and the C2 shape n = 8192, m = 16384) and each
leaf width, it reports the SYRK time (ev[1] -> ev[2] of the library, mean of --reps form + factor calls) of both paths,
and from one profiled call the time of each phase: the operand sums, the Winograd products (with their TFLOP/s),
the combination, the diagonal leaves and the scaled panel (which computes the column norms on the fast path).

    python scripts/fast_syrk_timing.py [--out DIR] [--reps 3] [--shapes 8192x131072,...] [--leaves 1024,2048,4096]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def phases_from_trace(path, depth):
    """Sum the kernel times of one form_H by phase.  fast_syrk_form launches, per depth, the sums, the products
    (one gemm_nt launch, perhaps followed by its split-K reduction) and the combination; then the leaves (the last
    gemm_nt launch).  So the first `depth` gemm_nt launches are products and the one after them the leaves."""
    with open(path) as f:
        ev = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    out = {"scale_panel": 0.0, "sums": 0.0, "products": 0.0, "combine": 0.0, "leaves": 0.0, "other": 0.0}
    gemms = 0
    for e in ev:
        name, ms = e["name"], e["dur"] / 1e3
        if "scale_panel" in name or "col_exponent" in name:
            out["scale_panel"] += ms
        elif "winograd_sums" in name:
            out["sums"] += ms
        elif "winograd_combine" in name:
            out["combine"] += ms
        elif "gemm_nt_kernel" in name or "splitk_reduce" in name:
            gemms += "gemm_nt_kernel" in name
            out["products" if gemms <= depth else "leaves"] += ms
        else:
            out["other"] += ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for the JSON lines (default: print only)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="8192x131072,12288x196608,16384x262144,8192x16384")
    ap.add_argument("--leaves", default="2048", help="leaf widths to sweep (CIP_FAST_SYRK_LEAF)")
    ap.add_argument("--leaf-sweep-n", type=int, default=16384, help="sweep --leaves only at this n (others: 2048)")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import conicip_b200 as cb
    from conicip_b200 import problems as P
    assert torch.cuda.is_available(), "needs a CUDA device"
    props = torch.cuda.get_device_properties(0)
    tmp = tempfile.mkdtemp(prefix="fast_syrk_timing_")
    lines = []

    def depth_of(n, leaf):
        W, depth = n, 0
        while W % 512 == 0 and W // 2 >= min(leaf, n // 2):
            W //= 2
            depth += 1
        return W, depth

    def run(n, m, fast, leaf):
        os.environ["CIP_FAST_SYRK"] = "1" if fast else "0"
        os.environ["CIP_FAST_SYRK_LEAF"] = str(leaf)
        pr = P.config4_device(n=n, m=m, seed=4)
        eng = cb.Engine(pr["Q"], pr["At"].t(), None, pr["cone_dims"])
        del pr
        torch.cuda.empty_cache()
        eng._bind_stream()
        g = torch.Generator(device="cuda")
        g.manual_seed(1)
        v = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
        s = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
        eng.nt_scaling(v, s)
        eng.form_H()                                   # warm-up (module load, tensor maps)
        torch.cuda.synchronize()
        syrk, scale = [], []
        for _ in range(args.reps):
            eng.factor_resident()                      # the library reads its SYRK events in factor_H
            torch.cuda.synchronize()
            st = eng.stats()
            syrk.append(st["ms_syrk"])
            scale.append(st["ms_scale"])
        trace = os.path.join(tmp, f"t_{n}_{m}_{int(fast)}_{leaf}.json")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.form_H()
            torch.cuda.synchronize()
        prof.export_chrome_trace(trace)
        ph = phases_from_trace(trace, depth_of(n, leaf)[1] if fast else 0)
        os.remove(trace)
        eng.close()
        del eng
        torch.cuda.empty_cache()
        return sum(syrk) / len(syrk), sum(scale) / len(scale), ph

    for shape in args.shapes.split(","):
        n, m = (int(x) for x in shape.split("x"))
        ms_c, sc_c, _ = run(n, m, False, 2048)
        leaves = [int(x) for x in args.leaves.split(",")] if n == args.leaf_sweep_n else [2048]
        for leaf in leaves:
            ms_f, sc_f, ph = run(n, m, True, leaf)
            # the products' flops: per depth d, 7 * 2^d products of (n / 2^(d+2))^2 outputs over m / 2 (2 flops each)
            W, depth = depth_of(n, leaf)
            K2 = ((m + 31) // 32 * 32 + 63) // 64 * 64 // 2
            pf = sum(7 * 2 ** d * (n >> (d + 2)) ** 2 * K2 * 2.0 for d in range(depth))
            rec = {"n": n, "m": m, "leaf": W, "depth": depth, "gpu": props.name,
                   "ms_syrk_classical": ms_c, "ms_syrk_fast": ms_f, "speedup": ms_c / ms_f,
                   "ms_scale_classical": sc_c, "ms_scale_fast": sc_f,
                   "phases_ms": ph, "products_tflops": pf / (ph["products"] * 1e-3) / 1e12 if ph["products"] else None,
                   "classical_tflops": m * float(n) * n / (ms_c * 1e-3) / 1e12,
                   "fast_effective_tflops": m * float(n) * n / (ms_f * 1e-3) / 1e12}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "fast_syrk_timing.jsonl"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
