"""CPU tests of the host-side logic: the F data carriers, cone-aligned row sharding, and the
N>1 path (partial Gram matrices + all-reduce) on gloo with world_size 2."""
import os
import socket

import numpy as np
import pytest

import oracle as O
from conicip_b200 import blocks as B
from conicip_b200 import problems as P
from conicip_b200.dist import shard_cones


def test_block_flatten_layout():
    F = B.Block([B.Diagonal([1.0, 2.0]), B.SymWoodbury([-3.0, 3.0, 3.0], [0.1, 0.2, 0.3], 1.0), B.Diagonal([5.0])])
    kind, fa, fb, fD, fR = F.flatten()
    assert kind.tolist() == [0, 1, 0] and kind.dtype == np.int32
    assert fa.tolist() == [1, 2, -3, 3, 3, 5] and fb.tolist() == [0, 0, 0.1, 0.2, 0.3, 0]
    assert fD.tolist() == [0, 1, 0] and fR is None and F.size == 6
    assert fa.flags.c_contiguous and fa.dtype == np.float64


def test_block_flatten_matches_oracle_nt_scaling():
    rng = np.random.default_rng(0)
    u = rng.standard_normal(4); z = np.concatenate([[np.linalg.norm(u) + 1], u])
    u = rng.standard_normal(4); s = np.concatenate([[np.linalg.norm(u) + 1], u])
    W = O.nestod_soc(z, s)
    kind, fa, fb, fD, _ = B.Block([B.SymWoodbury(W.Adiag, W.B, W.D)]).flatten()
    x = rng.standard_normal(5)
    assert np.allclose(fa * x + fD[0] * fb * (fb @ x), W.mul(x))


@pytest.mark.parametrize("cones,nr", [([("R", 100)], 4), ([("Q", 33)] * 8, 4), ([("R", 10), ("Q", 5), ("Q", 5), ("R", 7)], 2),
                                      ([("R", 262144)], 8), ([("Q", 7)] * 3, 8), ([("R", 5)], 1)])
def test_shard_cones_partitions_rows_on_cone_boundaries(cones, nr):
    sh = shard_cones(cones, nr)
    m = sum(k for _, k in cones)
    assert len(sh) == nr and sh[0][0] == 0 and sh[-1][1] == m
    for (lo, hi, cd), nxt in zip(sh, sh[1:] + [None]):
        assert sum(k for _, k in cd) == hi - lo
        if nxt:
            assert nxt[0] == hi
    # Q cones are never cut
    assert sorted(k for _, _, cd in sh for t, k in cd if t == "Q") == sorted(k for t, k in cones if t == "Q")
    if all(t == "R" for t, _ in cones) and m >= nr:
        sizes = [hi - lo for lo, hi, _ in sh]
        assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from conicip_b200.dist import TorchReducer
    prob = P.mixed(n=24, mr=20, ncones=4, k=5, p=0, seed=11)
    A, cd = prob["A"], prob["cone_dims"]
    lo, hi, lcd = shard_cones(cd, world)[rank]
    rng = np.random.default_rng(5)
    m = A.shape[0]
    v = np.zeros(m); s = np.zeros(m); off = 0
    for t, k in cd:
        if t == "R":
            v[off:off + k] = rng.uniform(0.5, 2, k); s[off:off + k] = rng.uniform(0.5, 2, k)
        else:
            for x in (v, s):
                u = rng.standard_normal(k - 1); x[off] = np.linalg.norm(u) + 0.5; x[off + 1:off + k] = u
        off += k

    def scaling(cdims, vv, ss):
        bl, o = [], 0
        for t, k in cdims:
            bl.append(O.Diag(np.sqrt(ss[o:o + k] / vv[o:o + k])) if t == "R" else O.nestod_soc(vv[o:o + k], ss[o:o + k]))
            o += k
        return O.Block(bl)

    Fl = scaling(lcd, v[lo:hi], s[lo:hi]).inv_adjoint()
    At = Fl.mul(A[lo:hi])
    Hpart = torch.from_numpy(At.T @ At + (prob["Q"] if rank == 0 else 0 * prob["Q"]))
    dist.all_reduce(Hpart)                                    # the engine does this with NCCL
    Ff = scaling(cd, v, s).inv_adjoint()
    Atf = Ff.mul(A)
    Hfull = prob["Q"] + Atf.T @ Atf
    red = TorchReducer()
    tot = red.sum(float(v[lo:hi] @ s[lo:hi]))
    mn = red.min(float(np.min(v[lo:hi])))
    tt = red.sum_tensor_(torch.tensor([float(v[lo:hi] @ s[lo:hi]), float(hi - lo)], dtype=torch.float64))
    ml = red.min_list([float(np.min(v[lo:hi])), float(rank)])
    ok = abs(float(tt[0]) - v @ s) < 1e-12 and float(tt[1]) == m and ml[0] == v.min() and ml[1] == 0.0
    q.put((rank, float(np.abs(Hpart.numpy() - Hfull).max()), abs(tot - v @ s), abs(mn - v.min()) + (0.0 if ok else 1.0)))
    dist.destroy_process_group()


def test_sharded_gram_allreduce_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, dh, ds, dm in res:
        assert dh < 1e-12 and ds < 1e-12 and dm == 0.0


def test_block_flatten_veccongurance():
    R = np.arange(9.0).reshape(3, 3)
    F = B.Block([B.Diagonal([1.0]), B.VecCongurance(R)])
    kind, fa, fb, fD, fR = F.flatten()
    assert kind.tolist() == [0, 2] and len(fa) == 1 + 6 and F.size == 7
    assert np.array_equal(fR, R.ravel(order="F"))            # column-major, as Julia's vec(R)


def test_julia_shim_binds_the_protocol_symbols():
    """The ccall shim a ConicIP.jl maintainer adds must name the same C symbols the header declares."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    jl = open(os.path.join(root, "conicip.jl_b200", "julia", "ConicIPB200.jl")).read()
    hdr = open(os.path.join(root, "include", "conicip_b200.h")).read()
    used = set(re.findall(r"\(:(cip_[a-z_0-9]+), LIB\)", jl))
    declared = set(re.findall(r"\b(cip_[a-z0-9_A-Z]+)\s*\(", re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)))
    assert used <= declared
    for s in ("cip_create", "cip_destroy", "cip_factor", "cip_solve", "cip_last_error"):
        assert s in used


def test_bench_reference_arm_schema():
    """`bench.py --impl reference` prints one JSON line with the contract's keys (tiny size here)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--n", "256", "--m", "1024",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in line
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_imcols_paths_that_need_no_device():
    """cip_imcols answers the empty matrix like the reference (src/preprocessor.jl:15: `([], true)`) and rejects
    bad arguments before touching CUDA, so both are checkable on the CPU box."""
    import ctypes as C

    import conicip_b200 as cb
    from conicip_b200._lib import lib, last_error

    R, ok = cb.imcols(np.zeros((0, 7)), np.zeros(0))
    assert ok and len(R) == 0
    R, ok = cb.imcols(np.zeros((3, 0)), np.zeros(3))
    assert ok and len(R) == 0
    keep = (C.c_int * 4)()
    nk, cons = C.c_int(0), C.c_int(0)
    A = np.zeros((4, 2))
    rc = lib().cip_imcols(-1, A.ctypes.data, 2, 4, 2, A.ctypes.data, 1e-8, keep, C.byref(nk), C.byref(cons))   # lda < p
    assert rc == -2 and "cip_imcols" in last_error()
    with pytest.raises(ValueError):
        cb.imcols(np.zeros((3, 2)), np.zeros(5))


def test_shard_plan_matches_python_mirror():
    """`cip_shard_plan` (what a handle with opts.ngpus = N does to the rows of A) is pure host logic and must
    agree with the Python mirror used by the one-process-per-GPU path (`dist.shard_cones`)."""
    import conicip_b200 as cb
    from conicip_b200.dist import shard_cones
    cases = [[("R", 1000)], [("R", 7)], [("Q", 33)] * 64, [("R", 80)] + [("Q", 9)] * 6,
             [("R", 20000), ("S", 2080)], [("Q", 5), ("R", 100), ("S", 21), ("Q", 40), ("R", 3)]]
    for cd in cases:
        m = sum(k for _, k in cd)
        for N in (1, 2, 3, 4, 8):
            plan = cb.shard_plan(cd, N)
            want = [(lo, hi) for lo, hi, _ in shard_cones(cd, N)]
            assert plan == want, (cd[:3], N, plan, want)
            assert plan[0][0] == 0 and plan[-1][1] == m
            assert all(plan[i][1] == plan[i + 1][0] for i in range(N - 1))
            # Q / S cones are never cut
            off = 0
            for t, k in cd:
                if t != "R":
                    assert any(lo <= off and off + k <= hi for lo, hi in plan), (t, k, plan)
                off += k


def _load_bench():
    import importlib.util
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    sys.modules["bench_mod"] = bench
    spec.loader.exec_module(bench)
    return bench


def test_bench_host_problem_c5_and_cpu_unit():
    """The host side of `bench.py --config C5` at a reduced size: the MOI-shaped LP with an S block of order 64, the
    synthetic interior points (S rows: vecm of a positive definite matrix) and one CPU unit through the oracle."""
    bench = _load_bench()
    prob, pts, rhs = bench.host_problem("C5", 2200, 2200 + 2080)
    assert prob["cone_dims"] == [("R", 2200), ("S", 2080)] and prob["A"].shape == (4280, 2200) and prob["G"].shape[0] > 0
    for v, s in pts:
        for x in (v, s):
            assert x[:2200].min() > 0 and np.linalg.eigvalsh(O.mat(x[2200:])).min() > 0
    assert len(rhs) == bench.NSOLVES
    assert 0 < bench.cpu_unit_oracle(prob, pts, rhs, repeats=1) < 120


def test_bench_dump_outputs_files_and_size_cap(tmp_path, monkeypatch):
    """`bench.py --dump-outputs DIR`: lambda and every solve's (dy, dv) as float64 .npy (an empty dw, p = 0, is left
    out); a vector over its share of the size cap becomes a sample that is the same in every run."""
    import types
    bench = _load_bench()
    D = types.SimpleNamespace(world=1, rank=0)
    rng = np.random.default_rng(3)
    lam = rng.standard_normal(1000)
    sols = [(rng.standard_normal(10), np.zeros(0), rng.standard_normal(1000)) for _ in range(bench.NSOLVES)]
    bench.dump_outputs(None, D, str(tmp_path / "a"), lam, sols)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == ["dv0", "dv1", "dy0", "dy1", "lambda"]
    assert all(x.dtype == np.float64 for x in got.values())
    assert np.array_equal(got["lambda"], lam) and np.array_equal(got["dv1"], sols[1][2])
    monkeypatch.setattr(bench, "DUMP_CAP_BYTES", 5 * 8 * 100)           # 100 entries for each of the 5 vectors
    for d in ("b", "c"):
        bench.dump_outputs(None, D, str(tmp_path / d), lam, sols)
    b, c = np.load(tmp_path / "b" / "lambda.npy"), np.load(tmp_path / "c" / "lambda.npy")
    assert len(b) == 100 and np.array_equal(b, c) and np.isin(b, lam).all()
    assert np.array_equal(np.load(tmp_path / "b" / "dy0.npy"), sols[0][0])


def test_ncu_traffic_table_matches_the_committed_captures():
    """`roofline.traffic` comes from profiles/ncu_traffic.json; every entry that names a committed raw ncu page must
    be reproducible from that page (scripts/ncu_traffic.py), i.e. the number is read from a capture, not typed in."""
    import importlib.util
    import json
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("ncu_traffic", os.path.join(root, "scripts", "ncu_traffic.py"))
    nt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(nt)
    tab = json.load(open(os.path.join(root, "profiles", "ncu_traffic.json")))
    checked = 0
    for key, ent in tab.items():
        m = re.match(r"(profiles/\S+_raw\.csv)", ent["source"])
        if not m:
            continue
        d = nt.read_raw(os.path.join(root, m.group(1)))[0]
        assert abs(d["dram__bytes_read.sum"] + d["dram__bytes_write.sum"] - ent["dram_bytes"]) <= 1e-6 * ent["dram_bytes"], key
        checked += 1
    assert checked >= 2 and "gemm_nt_syrk:n=16384,m=262144" in tab
