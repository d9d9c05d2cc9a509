"""`cip_options.row_structure`: singleton R rows on the diagonal of H, a compact SYRK for the other rows, and
Q + rho G'G formed once.  The reference for every comparison is the same library with the option off."""
import numpy as np
import pytest
import scipy.sparse as sp

import conicip_b200 as cb
from conicip_b200 import problems as P

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _option_decides(monkeypatch):
    # CIP_ROW_STRUCTURE=1 would turn the reference engines (row_structure=0) structured as well
    monkeypatch.delenv("CIP_ROW_STRUCTURE", raising=False)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def interior(cone_dims, seed=0):
    """A strictly interior pair (v, s) of the cone product."""
    rng = np.random.default_rng(seed)
    vs = []
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
        vs.append(np.concatenate(x))
    return vs


def engines(prob, A=None, **kw):
    G = prob["G"] if prob["G"].shape[0] else None
    A = prob["A"] if A is None else A
    return (cb.Engine(prob["Q"], A, G, prob["cone_dims"], row_structure=1, **kw),
            cb.Engine(prob["Q"], A, G, prob["cone_dims"], row_structure=0, **kw))


def unit(e, v, s, rng):
    """form H at the NT scaling of (v, s), then factor and solve one right-hand side"""
    lam = e.nt_scaling(v, s)
    e.form_H()
    H = np.tril(e.get_H())
    e.factor_H()
    ry, rw, rv = rng.standard_normal(e.n), rng.standard_normal(e.p), rng.standard_normal(e.m)
    return lam, H, e.solve(ry, rw if e.p else None, rv)


def compare_units(e_on, e_off, cone_dims, tol_H=1e-13, tol_solve=1e-12):
    v, s = interior(cone_dims)
    _, Hon, son = unit(e_on, v, s, np.random.default_rng(1))
    _, Hoff, soff = unit(e_off, v, s, np.random.default_rng(1))
    assert np.abs(Hon - Hoff).max() / np.linalg.norm(Hoff) < tol_H
    for a, b in zip(son, soff):
        if len(b):
            assert rel(a, b) < tol_solve


def mixed_problem(seed=11, n=120, p=7):
    """R rows with 0, 1 and >= 2 non-zeros interleaved in one R cone, a Q cone whose rows are singletons, a Q cone
    of dense rows, one S cone, equalities; strictly feasible, Q positive definite."""
    rng = np.random.default_rng(seed)
    rows, cones = [], []
    kinds = np.tile([0, 1, 2, 1, 1, 2], 10)               # 60 R rows
    for kd in kinds:
        a = np.zeros(n)
        if kd == 1:
            a[rng.integers(n)] = rng.choice([-1.0, 1.0]) * rng.uniform(0.5, 2.0)
        elif kd == 2:
            idx = rng.choice(n, 6, replace=False)
            a[idx] = rng.standard_normal(6)
        rows.append(a)
    cones.append(("R", len(kinds)))
    for j in rng.choice(n, 4, replace=False):            # Q cone of singleton rows: stays in the rest
        a = np.zeros(n)
        a[j] = 1.0
        rows.append(a)
    cones.append(("Q", 4))
    rows.extend(rng.standard_normal((5, n)) / np.sqrt(n))
    cones.append(("Q", 5))
    rows.extend(rng.standard_normal((6, n)) / np.sqrt(n))  # S cone of order 3
    cones.append(("S", 6))
    A = np.array(rows)
    y0 = rng.standard_normal(n)
    v0, _ = interior(cones, seed)
    b = A @ y0 - v0
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    d = G @ y0
    Q = P._lowrank_q(rng, n, 8)
    c = rng.standard_normal(n)
    return P._prob("mixed_rows", Q, c, A, b, cones, G, d, optTol=1e-8)


def with_explicit_zero(A):
    """CSC copy of A with one explicitly stored zero (in an empty row) and one in a singleton row"""
    C = sp.coo_matrix(A)
    zr = np.where(~A.any(axis=1))[0][0]
    sr = np.where((A != 0).sum(axis=1) == 1)[0][0]
    sc = int(np.where(A[sr] == 0)[0][0])
    M = sp.csc_matrix((np.concatenate([C.data, [0.0, 0.0]]), (np.concatenate([C.row, [zr, sr]]),
                                                                  np.concatenate([C.col, [0, sc]]))), shape=A.shape)
    assert (M.data == 0).sum() == 2
    return M


# ---------------------------------------------------------------- 1. A = [I; -I] and A = I
@pytest.mark.parametrize("make", [lambda: P.box_qp(300), lambda: P.box_qp(1000), lambda: P.config1(500),
                                  lambda: P.config1(1000)], ids=["box300", "box1000", "c1_500", "c1_1000"])
def test_all_singleton_rows(make):
    prob = make()
    e_on, e_off = engines(prob)
    info = e_on.structure_info()
    assert info["enabled"] == 1 and info["rest_rows"] == 0
    assert info["singleton_rows"] == e_on.m and info["empty_rows"] == 0
    assert e_off.structure_info()["enabled"] == 0
    compare_units(e_on, e_off, prob["cone_dims"])
    assert e_on.stats()["syrk_flops"] == 0
    r_on = e_on.ipm_solve(prob["c"], prob["b"], None, optTol=1e-8)
    r_off = e_off.ipm_solve(prob["c"], prob["b"], None, optTol=1e-8)
    assert r_on[3]["status"] == r_off[3]["status"] == "Optimal"
    assert r_on[3]["Iter"] == r_off[3]["Iter"]
    assert rel(r_on[0], r_off[0]) < 1e-8 and rel(r_on[2], r_off[2]) < 1e-8
    e_on.close(); e_off.close()


# ---------------------------------------------------------------- 2. C5-shaped
def test_c5_shaped_compressed_with_constant_base():
    prob = P.config5(n=2200, k=32, p=100)
    e_on, e_off = engines(prob)
    info = e_on.structure_info()
    dim = 32 * 33 // 2
    assert info == dict(enabled=1, singleton_rows=2200, empty_rows=0, rest_rows=dim, rest_cols=dim, compressed=1,
                        base_has_gtg=1)
    compare_units(e_on, e_off, prob["cone_dims"])
    assert e_on.stats()["syrk_flops"] == dim ** 3
    # 7. the compact copy of A and no dense Atil: fewer resident bytes
    assert e_on.stats()["device_bytes"] < e_off.stats()["device_bytes"]
    r_on = e_on.ipm_solve(prob["c"], prob["b"], prob["d"], optTol=1e-8)
    r_off = e_off.ipm_solve(prob["c"], prob["b"], prob["d"], optTol=1e-8)
    assert r_on[3]["status"] == r_off[3]["status"] == "Optimal"
    assert abs(r_on[3]["Iter"] - r_off[3]["Iter"]) <= 1
    for a, b in zip(r_on[:3], r_off[:3]):
        assert rel(a, b) < 1e-6
    e_on.close(); e_off.close()


# ---------------------------------------------------------------- 3. mixed rows, dense and CSC input
def test_mixed_rows_dense_and_csc_agree_bitwise():
    prob = mixed_problem()
    A = prob["A"]
    e_dense, e_off = engines(prob)
    e_csc = cb.Engine(sp.csc_matrix(prob["Q"]), with_explicit_zero(A), sp.csc_matrix(prob["G"]), prob["cone_dims"],
                      row_structure=1)
    info = e_dense.structure_info()
    assert info == e_csc.structure_info()
    assert info["singleton_rows"] == 30 and info["empty_rows"] == 10
    assert info["rest_rows"] == 20 + 4 + 5 + 6 and info["compressed"] == 0 and info["base_has_gtg"] == 1
    rng = np.random.default_rng(2)
    x, u = rng.standard_normal(e_dense.n), rng.standard_normal(e_dense.m)
    for e in (e_dense, e_csc):
        assert rel(e.mul_A(x), A @ x) < 1e-14
        assert rel(e.mul_A(u, trans=True), A.T @ u) < 1e-14
    assert np.array_equal(e_dense.mul_A(x), e_csc.mul_A(x))
    assert np.array_equal(e_dense.mul_A(u, trans=True), e_csc.mul_A(u, trans=True))
    v, s = interior(prob["cone_dims"])
    _, Hd, sd = unit(e_dense, v, s, np.random.default_rng(3))
    _, Hc, sc = unit(e_csc, v, s, np.random.default_rng(3))
    assert np.array_equal(Hd, Hc)
    for a, b in zip(sd, sc):
        assert np.array_equal(a, b)
    compare_units(e_dense, e_off, prob["cone_dims"])
    e_dense.close(); e_csc.close(); e_off.close()


# ---------------------------------------------------------------- 4. nothing to exploit: bit-identical
def test_no_singletons_no_equalities_is_bit_identical():
    prob = P.config2(n=640, m=1200)
    e_on, e_off = engines(prob)
    info = e_on.structure_info()
    assert info["rest_rows"] == 1200 and info["singleton_rows"] == 0 and info["compressed"] == 0
    v, s = interior(prob["cone_dims"])
    _, Hon, son = unit(e_on, v, s, np.random.default_rng(4))
    _, Hoff, soff = unit(e_off, v, s, np.random.default_rng(4))
    assert np.array_equal(Hon, Hoff)
    for a, b in zip(son, soff):
        assert np.array_equal(a, b)
    e_on.close(); e_off.close()


# ---------------------------------------------------------------- 5. full-width folded rest
def test_bounds_plus_dense_rows_folded_rest():
    rng = np.random.default_rng(5)
    base = P.config2(n=512, m=700, seed=6)
    n = 512
    A = np.vstack([base["A"], np.eye(n)])
    y0 = rng.uniform(0.5, 1.5, n)
    s0 = rng.uniform(0.1, 1.1, A.shape[0])
    prob = P._prob("c2_bounds", base["Q"], base["c"], A, A @ y0 - s0, [("R", A.shape[0])], optTol=1e-8)
    e_on, e_off = engines(prob, fold_scaling=1)
    info = e_on.structure_info()
    assert info["singleton_rows"] == n and info["rest_rows"] == 700 and info["rest_cols"] == n
    assert info["compressed"] == 0
    compare_units(e_on, e_off, prob["cone_dims"])
    e_on.close(); e_off.close()


# ---------------------------------------------------------------- 6. determinism, cip_solve_multi
def test_deterministic_and_solve_multi_matches_solve():
    prob = P.config5(n=2200, k=32, p=100)
    e = engines(prob)[0]
    v, s = interior(prob["cone_dims"])
    runs = [unit(e, v, s, np.random.default_rng(6)) for _ in range(2)]
    for a, b in zip(runs[0][2], runs[1][2]):
        assert np.array_equal(a, b)
    assert np.array_equal(runs[0][1], runs[1][1])
    rng = np.random.default_rng(7)
    k = 3
    RY, RW, RV = rng.standard_normal((e.n, k)), rng.standard_normal((e.p, k)), rng.standard_normal((e.m, k))
    DY, DW, DV = e.solve_multi(np.asfortranarray(RY), np.asfortranarray(RW), np.asfortranarray(RV))
    for j in range(k):
        dy, dw, dv = e.solve(RY[:, j].copy(), RW[:, j].copy(), RV[:, j].copy())
        assert np.array_equal(DY[:, j], dy) and np.array_equal(DW[:, j], dw) and np.array_equal(DV[:, j], dv)
    e.close()


# ---------------------------------------------------------------- 8. sharded handles refuse it
def test_sharded_handle_is_rejected():
    prob = P.box_qp(64)
    for A in (prob["A"], sp.csc_matrix(prob["A"])):
        with pytest.raises(cb.CipError, match="single-device"):
            cb.Engine(prob["Q"], A, None, prob["cone_dims"], ngpus=2, row_structure=1)


# ---------------------------------------------------------------- 9. the host-driven loop on top
def test_host_driven_conicip_matches_native():
    prob = mixed_problem()
    args = (prob["Q"], prob["c"], prob["A"], prob["b"], prob["cone_dims"], prob["G"], prob["d"])
    s_host = cb.conicIP(*args, kktsolver=cb.make_kktsolver(row_structure=1), optTol=1e-8)
    s_nat = cb.conicIP_native(*args, row_structure=1, optTol=1e-8)
    s_off = cb.conicIP_native(*args, optTol=1e-8)
    assert s_host.status == s_nat.status == s_off.status == "Optimal"
    assert abs(s_host.Iter - s_nat.Iter) <= 1
    for f in ("y", "w", "v"):
        assert rel(getattr(s_host, f), getattr(s_nat, f)) < 1e-6
        assert rel(getattr(s_nat, f), getattr(s_off, f)) < 1e-6
