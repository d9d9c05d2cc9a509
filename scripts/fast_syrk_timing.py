"""Phase timing of the fast SYRK of form_H (csrc/fast_syrk.cu) against the classical SYRK, on the device-generated
dense QP of bench.py (problems.config4_device, all rows R).

For each shape (default n in {8192, 12288, 16384} with m = 16 n, and the C2 shape n = 8192, m = 16384), each
leaf width and each level setting (CIP_FAST_SYRK_LEVELS: 1 = one Winograd level everywhere, 2 = two wherever the
tiles allow it, 0 = the library's rule), it reports the SYRK time (ev[1] -> ev[2] of the library, mean of --reps
form + factor calls) of both paths, and from one profiled call the time of each phase: the level-1 and level-2
operand sums, the products of each level (with their TFLOP/s), the two combinations, the diagonal leaves and the
scaled panel (which computes the column norms on the fast path).

    python scripts/fast_syrk_timing.py [--out DIR] [--reps 3] [--shapes 8192x131072,...] [--leaves 1024,2048,4096]
                                       [--levels 1,2]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


PHASES = ("scale_panel", "sums", "sums2", "products", "products2", "combine", "combine2", "leaves", "other")
DEPTH_PHASES = ("sums", "sums2", "products", "products2", "combine2", "combine")


def classify(events):
    """Sum kernel times by phase, by kernel name, in total and per depth.  gemm_nt launches (and their split-K
    reductions) take the phase of the combination that reads them: the level-1 products precede
    winograd_combine_kernel, the level-2 products winograd_combine2_kernel, and the leaves, launched last, precede
    none.  Each winograd_combine_kernel closes one depth; a depth with winograd_combine2_kernel launches took two
    levels (read from what ran, so a handle that fell back to one level for lack of memory reports one)."""
    out = {k: 0.0 for k in PHASES}
    depths, cur = [], {k: 0.0 for k in DEPTH_PHASES}
    pending = 0.0

    def add(k, ms):
        out[k] += ms
        if k in cur:
            cur[k] += ms

    for e in sorted(events, key=lambda e: e["ts"]):
        name, ms = e["name"], e["dur"] / 1e3
        if "gemm_nt_kernel" in name or "splitk_reduce" in name:
            pending += ms
            continue
        if "scale_panel" in name or "col_exponent" in name:
            add("scale_panel", ms)
        elif "winograd_sums2" in name:
            add("sums2", ms)
        elif "winograd_sums" in name:
            add("sums", ms)
        elif "winograd_combine2" in name:
            add("combine2", ms)
            add("products2", pending)
            pending = 0.0
        elif "winograd_combine" in name:
            add("combine", ms)
            add("products", pending)
            pending = 0.0
            depths.append(cur)
            cur = {k: 0.0 for k in DEPTH_PHASES}
        else:
            add("other", ms)
    add("leaves", pending)
    for d in depths:
        d["levels"] = 2 if d["combine2"] > 0 else 1
        d["ms"] = sum(d[k] for k in DEPTH_PHASES)
    return out, depths


def phases_from_trace(path):
    with open(path) as f:
        return classify([e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"])


def depth_of(n, leaf):
    """fast_syrk_plan's halving with CIP_FAST_SYRK=1: (leaf width, depth)."""
    W, depth = n, 0
    while W % 512 == 0 and W // 2 >= min(leaf, n // 2):
        W //= 2
        depth += 1
    return W, depth


def depth_flops(n, m, d, levels, any_two):
    """Flops (2 per multiply-add) of the products of depth d: 7 * 2^d products of (n / 2^(d+2))^2 outputs over K2,
    or, at two levels, 49 * 2^d of (n / 2^(d+3))^2 over K2 / 2.  K2 is rounded to 64 when any depth takes two."""
    q = 128 if any_two else 64
    K2 = ((m + 31) // 32 * 32 + q - 1) // q * q // 2
    if levels == 2:
        return 49 * 2 ** d * (n >> (d + 3)) ** 2 * (K2 // 2) * 2.0
    return 7 * 2 ** d * (n >> (d + 2)) ** 2 * K2 * 2.0


def selftest():
    """The argument parsing and the trace classifier on a synthetic trace (no device needed)."""
    ev, t = [], 0
    for name, dur in [("scale_panel_diag_norms_kernel", 5), ("col_exponent_kernel", 1), ("winograd_sums_kernel", 7),
                      ("winograd_sums2_kernel", 2), ("gemm_nt_kernel<false>", 100), ("splitk_reduce_kernel", 1),
                      ("winograd_combine2_kernel", 3), ("winograd_sums2_kernel", 2), ("gemm_nt_kernel<false>", 100),
                      ("winograd_combine2_kernel", 3), ("winograd_combine_kernel", 4), ("winograd_sums_kernel", 7),
                      ("gemm_nt_kernel<false>", 50), ("winograd_combine_kernel", 4), ("gemm_nt_kernel<false>", 30),
                      ("splitk_reduce_kernel", 1)]:
        ev.append({"name": name, "ts": t, "dur": dur * 1e3})
        t += dur + 1
    ph, depths = classify(list(reversed(ev)))
    want = {"scale_panel": 6, "sums": 14, "sums2": 4, "products": 50, "products2": 201, "combine": 8, "combine2": 6,
            "leaves": 31, "other": 0}
    assert ph == {k: float(v) for k, v in want.items()}, ph
    assert [d["levels"] for d in depths] == [2, 1], depths
    assert depths[0]["ms"] == 7 + 4 + 201 + 6 + 4 and depths[1]["ms"] == 7 + 50 + 4, depths
    assert parse_args(["--levels", "1,2"]).levels == "1,2"
    print("selftest ok")


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="directory for the JSON lines (default: print only)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="8192x131072,12288x196608,16384x262144,8192x16384")
    ap.add_argument("--leaves", default="2048", help="leaf widths to sweep (CIP_FAST_SYRK_LEAF)")
    ap.add_argument("--leaf-sweep-n", type=int, default=16384, help="sweep --leaves only at this n (others: 2048)")
    ap.add_argument("--levels", default="0", help="CIP_FAST_SYRK_LEVELS settings to sweep (0: the library's rule)")
    ap.add_argument("--selftest", action="store_true", help="check the trace classifier on a synthetic trace and exit")
    return ap.parse_args(argv)


def main():
    args = parse_args()
    if args.selftest:
        selftest()
        return

    import torch
    from torch.profiler import ProfilerActivity, profile

    import conicip_b200 as cb
    from conicip_b200 import problems as P
    assert torch.cuda.is_available(), "needs a CUDA device"
    props = torch.cuda.get_device_properties(0)
    tmp = tempfile.mkdtemp(prefix="fast_syrk_timing_")
    lines = []

    def run(n, m, fast, leaf, levels=0):
        os.environ["CIP_FAST_SYRK"] = "1" if fast else "0"
        os.environ["CIP_FAST_SYRK_LEAF"] = str(leaf)
        os.environ["CIP_FAST_SYRK_LEVELS"] = str(levels)
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
        dev_bytes = st["device_bytes"]
        trace = os.path.join(tmp, f"t_{n}_{m}_{int(fast)}_{leaf}.json")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.form_H()
            torch.cuda.synchronize()
        prof.export_chrome_trace(trace)
        ph = phases_from_trace(trace)
        os.remove(trace)
        eng.close()
        del eng
        torch.cuda.empty_cache()
        return sum(syrk) / len(syrk), sum(scale) / len(scale), ph, dev_bytes

    for shape in args.shapes.split(","):
        n, m = (int(x) for x in shape.split("x"))
        ms_c, sc_c, _, bytes_c = run(n, m, False, 2048)
        leaves = [int(x) for x in args.leaves.split(",")] if n == args.leaf_sweep_n else [2048]
        for leaf in leaves:
            for levels in (int(x) for x in args.levels.split(",")):
                ms_f, sc_f, (ph, depths), bytes_f = run(n, m, True, leaf, levels)
                W, depth = depth_of(n, leaf)
                two = [d for d, x in enumerate(depths) if x["levels"] == 2]
                f1 = f2 = 0.0
                for d, x in enumerate(depths):
                    f = depth_flops(n, m, d, x["levels"], bool(two))
                    x["products_tflops"] = f / ((x["products"] + x["products2"]) * 1e-3) / 1e12
                    if x["levels"] == 2:
                        f2 += f
                    else:
                        f1 += f
                rec = {"n": n, "m": m, "leaf": W, "depth": depth, "levels": levels, "two_level_depths": two,
                       "gpu": props.name, "ms_syrk_classical": ms_c, "ms_syrk_fast": ms_f, "speedup": ms_c / ms_f,
                       "ms_scale_classical": sc_c, "ms_scale_fast": sc_f, "phases_ms": ph, "per_depth_ms": depths,
                       "products_tflops": f1 / (ph["products"] * 1e-3) / 1e12 if ph["products"] else None,
                       "products2_tflops": f2 / (ph["products2"] * 1e-3) / 1e12 if ph["products2"] else None,
                       "classical_tflops": m * float(n) * n / (ms_c * 1e-3) / 1e12,
                       "fast_effective_tflops": m * float(n) * n / (ms_f * 1e-3) / 1e12,
                       "device_bytes_classical": bytes_c, "device_bytes_fast": bytes_f}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "fast_syrk_timing.jsonl"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
