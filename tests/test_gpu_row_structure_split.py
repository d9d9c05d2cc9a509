"""`cip_options.row_structure = 2`: H factored as its diagonal on the columns D plus the dense block H_KK on the
coupled columns K, with no n_pad x n_pad buffer.

References: the FP64 evaluation of H and its rounding-error bound from test_gpu_row_structure_reference.py (imported,
not copied), the oracle's KKT solvers, the same library in mode 1, and NumPy / scipy.sparse on the host.  The mirror
of the column rule and the sparse C5 generator run without a GPU.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
from conicip_b200 import problems as P
from test_gpu_row_structure_reference import (C_H, U, assert_H, check_solve, cone_point, dense, oracle_F, ref_H,
                                              rel, round_up, sparse_row)


@pytest.fixture(autouse=True)
def _option_decides(monkeypatch):
    # CIP_ROW_STRUCTURE would override the row_structure each engine here is created with
    monkeypatch.delenv("CIP_ROW_STRUCTURE", raising=False)


# ================================================================ the mirror of the column rule
def rest_columns(A, cone_dims):
    """J of mode 1: the columns touched by a Q / S row or an R row with >= 2 non-zeros (-0.0 is zero)."""
    A = dense(A, None)
    nz = A != 0.0
    is_r = np.concatenate([np.full(k, t == "R") for t, k in cone_dims])
    rest = ~is_r | (nz.sum(axis=1) >= 2)
    return nz[rest].any(axis=0)


def expected_split_info(Q, A, G, cone_dims, aug_rho=-1.0):
    """K = J, plus every column with an off-diagonal non-zero of Q in its row or its column, plus -- when the resolved
    rho > 0 and p > 0 -- every column where G has a non-zero.  Q and G are taken after duplicates are summed (a
    scipy matrix is densified, which sums them); a non-zero is a value != 0.0.  D is the rest."""
    A = dense(A, None)
    m, n = A.shape
    if m == 0:
        return dict(enabled=0, coupled_cols=0, diagonal_cols=0, cols_from_rest=0, cols_from_Q=0, cols_from_G=0)
    J = rest_columns(A, cone_dims)
    Qd = dense(Q, (n, n)) if Q is None or sp.issparse(Q) or np.ndim(Q) == 2 else np.diag(Q)
    off = (Qd != 0.0) & ~np.eye(n, dtype=bool)
    Kq = off.any(axis=0) | off.any(axis=1)
    Gd = dense(G, (0, n))
    p = Gd.shape[0]
    rho = (aug_rho if aug_rho >= 0 else 1.0) if p > 0 else 0.0
    Kg = (Gd != 0.0).any(axis=0) if rho > 0 else np.zeros(n, dtype=bool)
    K = J | Kq | Kg
    return dict(enabled=1, coupled_cols=int(K.sum()), diagonal_cols=int(n - K.sum()), cols_from_rest=int(J.sum()),
                cols_from_Q=int(Kq.sum()), cols_from_G=int(Kg.sum()))


def mirror_problem():
    """n = 12: column 0..1 in a rest row; Q couples 3-4 (symmetric), 6 (asymmetric: Q[6, 9] only, so 9 too);
    G touches 10 and 11; a stored -0.0 at Q[7, 8]; singletons on the others."""
    n = 12
    A = np.zeros((n + 1, n))
    A[0, 0], A[0, 1] = 1.0, 2.0
    for j in range(n):
        A[1 + j, j] = 1.0
    Q = np.eye(n)
    Q[3, 4] = Q[4, 3] = 0.5
    Q[6, 9] = 0.25
    Q[7, 8] = -0.0
    G = np.zeros((1, n))
    G[0, 10], G[0, 11] = 1.0, -1.0
    return Q, A, G, [("R", n + 1)]


def test_split_mirror_on_hand_counted_cases():
    Q, A, G, cd = mirror_problem()
    assert expected_split_info(Q, A, G, cd) == dict(enabled=1, coupled_cols=8, diagonal_cols=4, cols_from_rest=2,
                                                    cols_from_Q=4, cols_from_G=2)
    assert expected_split_info(Q, A, G, cd, aug_rho=0.0)["coupled_cols"] == 6
    assert expected_split_info(np.diag(Q).copy(), A, G, cd, aug_rho=0.0)["cols_from_Q"] == 0       # diagonal Q
    assert expected_split_info(None, A, G, cd, aug_rho=0.0)["coupled_cols"] == 2                    # no Q
    # CSC with duplicates that cancel off the diagonal: no coupling; one that does not cancel: coupling
    Qs = sp.csc_matrix((np.array([1.0, 0.5, -0.5, 1.0]), (np.array([0, 5, 5, 2]), np.array([0, 2, 2, 2]))),
                       shape=(12, 12))
    assert expected_split_info(Qs, A, None, cd)["cols_from_Q"] == 0
    Qs2 = sp.csc_matrix((np.array([0.5, 0.25]), (np.array([5, 5]), np.array([2, 2]))), shape=(12, 12))
    assert expected_split_info(Qs2, A, None, cd)["cols_from_Q"] == 2


def test_config5_sparse_equals_config5():
    a, b = P.config5(n=700, k=8, p=30, seed=9), P.config5_sparse(n=700, k=8, p=30, seed=9)
    assert a["cone_dims"] == b["cone_dims"]
    for key in ("A", "G", "Q"):
        assert sp.issparse(b[key]) and np.array_equal(a[key], b[key].toarray()), key
    assert np.array_equal(a["c"], b["c"]) and np.array_equal(a["b"], b["b"])
    # d = G y0: the dense and the sparse product sum the ten terms of a row in different orders
    assert np.abs(a["d"] - b["d"]).max() <= 1e-13 * (1 + np.abs(a["d"]).max())


# ================================================================ problems
def split_problem(seed=31, n=300, p=5):
    """Both D and K non-empty: dense Q with a few off-diagonal pairs, singletons on D and on K columns, R rest rows
    with >= 2 non-zeros, a Q cone and an S cone over a scattered column set, sparse equality rows (so at rho = 0
    some G columns lie in D), and column n-1 touched by Q_jj alone.  Strictly feasible, Q positive definite."""
    rng = np.random.default_rng(seed)
    Jc = np.sort(rng.choice(n - 1, 40, replace=False))
    Q = np.diag(rng.uniform(0.5, 2.0, n))
    for a, b in ((10, 250), (40, 41), (127, 128), (3, 200)):
        Q[a, b] = Q[b, a] = 0.2
    rows = []
    for j in range(n - 1):
        if j % 3 != 2:                           # every third column has no bound
            rows.append(sparse_row(n, [j], rng))
        if j % 25 == 0:
            rows.append(sparse_row(n, rng.choice(Jc, 3, replace=False), rng))
    cones = [("R", len(rows))]
    rows += [sparse_row(n, rng.choice(Jc, 6, replace=False), rng) / 4 for _ in range(5)]
    cones.append(("Q", 5))
    rows += [sparse_row(n, rng.choice(Jc, 2, replace=False), rng) for _ in range(6)]
    cones.append(("S", 6))
    A = np.array(rows)
    G = np.zeros((p, n))
    for i in range(p):
        G[i, rng.choice(n - 1, 4, replace=False)] = rng.standard_normal(4)
    y0 = rng.standard_normal(n)
    b = A @ y0 - cone_point(cones, rng)
    return P._prob("split_mixed", Q, rng.standard_normal(n), A, b, cones, G, G @ y0, optTol=1e-8)


def coupled_everywhere_problem(p, full_rest, seed=32, n=256):
    """D is empty: a dense low-rank Q couples every column.  The rest is a few sparse rows (mode 1 compresses it)
    or rows over every column (mode 1 runs the SYRK on all columns)."""
    rng = np.random.default_rng(seed)
    rows = [sparse_row(n, [j], rng) for j in range(n)]
    cols = lambda: np.arange(n) if full_rest else rng.choice(n, 4, replace=False)
    rows += [sparse_row(n, cols(), rng) / 4 for _ in range(12)]
    cones = [("R", n + 12)]
    rows += [sparse_row(n, cols(), rng) / 8 for _ in range(4)]
    cones.append(("Q", 4))
    A = np.array(rows)
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    y0 = rng.standard_normal(n)
    b = A @ y0 - cone_point(cones, rng)
    return P._prob("coupled", P._lowrank_q(rng, n, 8), rng.standard_normal(n), A, b, cones, G, G @ y0)


def engine(prob, mode=2, A=None, Q="prob", **kw):
    import conicip_b200 as cb
    G = prob["G"] if prob["G"].shape[0] else None
    return cb.Engine(prob["Q"] if isinstance(Q, str) else Q, prob["A"] if A is None else A, G, prob["cone_dims"],
                     row_structure=mode, **kw)


def rho_of(prob, aug_rho):
    return (aug_rho if aug_rho >= 0 else 1.0) if prob["G"].shape[0] else 0.0


def assert_LLt(L, ref, what=""):
    """L L' against the reference H: the bound of H plus the backward error of a Cholesky factorisation,
    |L L' - H| <= gamma_{n+1} |L| |L'| (Higham, Accuracy and Stability, thm. 10.3), with the same constant C_H."""
    n = L.shape[0]
    tol = C_H * U * (ref.k + 2) * ref.B + C_H * U * (n + 2) * (np.abs(L) @ np.abs(L).T)
    bad = np.tril(~(np.abs(L @ L.T - ref.H) <= tol))
    assert not bad.any(), f"{what}: L L' differs from H at {np.argwhere(bad)[0]}"


def check_split_H(e, prob, seed, aug_rho=-1.0, delta=0.0):
    """H at a wide and at a central scaling before the factorisation, L L' after it; returns (F, ref) of the
    central point, whose scaling stays resident"""
    rng = np.random.default_rng(seed)
    cd = prob["cone_dims"]
    for wide in (True, False):
        v, s = cone_point(cd, rng, wide), cone_point(cd, rng, wide)
        e.nt_scaling(v, s)
        e.form_H()
        Fo = oracle_F(cd, v, s)
        ref = ref_H(prob["Q"], prob["A"], prob["G"], cd, Fo, rho_of(prob, aug_rho), delta)
        what = "wide" if wide else "central"
        assert_H(e.get_H(), ref, what)
        assert e.factor_H() == 0
        assert_LLt(np.tril(e.get_H()), ref, what)
    e.form_H()                           # the resident H again (check_solve factors it)
    return Fo, ref, (v, s)


# ================================================================ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["dense_q0", "diag_q1", "csc_q2", "csc_cancel", "negzero", "asym", "rho0"])
def test_split_info_matches_mirror(variant):
    import conicip_b200 as cb
    Q, A, G, cd = mirror_problem()
    kw, Qin, Ain = {}, Q, A
    if variant == "diag_q1":
        Qin = sp.diags(np.diag(Q)).tocsc()         # the Engine passes a diagonal matrix as q_kind = 1
    elif variant == "csc_q2":
        Qin, Ain = sp.csc_matrix(Q), sp.csc_matrix(A)
    elif variant == "csc_cancel":
        Ain = sp.csc_matrix(A)
        Qin = Q.copy()
        Qin[3, 4] = Qin[4, 3] = Qin[6, 9] = 0.0
        # duplicates summing to 0 at (5, 2) and (2, 5): stored zeros after summation, no coupling
        Qin = sp.csc_matrix((np.concatenate([np.diag(Q), [0.5, -0.5, 0.5, -0.5]]),
                             (np.concatenate([np.arange(12), [5, 5, 2, 2]]), np.concatenate([np.arange(12), [2, 2, 5, 5]]))),
                            shape=(12, 12))
    elif variant == "negzero":
        Qin = Q.copy()
        Qin[3, 4] = Qin[4, 3] = -0.0
        Qin[6, 9] = 0.0
    elif variant == "asym":
        Qin = Q.copy()
        Qin[3, 4] = Qin[4, 3] = 0.0                # only Q[6, 9]: couples 6 and 9
    elif variant == "rho0":
        kw["aug_rho"] = 0.0
    e = cb.Engine(Qin, Ain, G, cd, row_structure=2, **kw)
    want = expected_split_info(Qin, A, G, cd, kw.get("aug_rho", -1.0))
    assert e.split_info() == want
    assert e.structure_info()["compressed"] == 1
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("aug_rho", [-1.0, 0.0])
@pytest.mark.parametrize("csc", [False, True])
def test_mixed_split_against_reference(aug_rho, csc):
    prob = split_problem()
    A = sp.csc_matrix(prob["A"]) if csc else prob["A"]
    Q = sp.csc_matrix(prob["Q"]) if csc else prob["Q"]
    e = engine(prob, A=A, Q=Q, aug_rho=aug_rho)
    info = e.split_info()
    assert info == expected_split_info(prob["Q"], prob["A"], prob["G"], prob["cone_dims"], aug_rho)
    assert 0 < info["coupled_cols"] < len(prob["c"])
    Fo, ref, (v, s) = check_split_H(e, prob, 5, aug_rho=aug_rho)
    rng = np.random.default_rng(6)
    dy, dw, dv = check_solve(e, prob, Fo, ref, rng)
    # mode 1 solves the same system through the dense H.  Both are backward stable, so they differ by at most
    # about cond(KKT) * n * u; at the central point the oracle comparison inside check_solve already holds both to
    # 1e-9 of the exact solution, so 2e-9 between the modes is the same statement, not a looser one.
    e1 = engine(prob, mode=1, A=A, Q=Q, aug_rho=aug_rho)
    e1.nt_scaling(v, s)
    e1.form_H()
    y1, w1, v1 = check_solve(e1, prob, Fo, ref, np.random.default_rng(6))
    assert rel(dy, y1) < 2e-9 and rel(dv, v1) < 2e-9 and rel(dw, w1) < 2e-9
    e1.close()
    e.close()


@pytest.mark.gpu
def test_mixed_split_with_reg_delta():
    prob = split_problem(seed=33)
    e = engine(prob, reg_delta=1e-3)
    check_split_H(e, prob, 7, delta=1e-3)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("p,full_rest", [(0, False), (5, False), (5, True)])
def test_no_diagonal_columns_is_bit_identical_to_mode_1(p, full_rest):
    prob = coupled_everywhere_problem(p, full_rest)
    e2, e1 = engine(prob), engine(prob, mode=1)
    assert e2.split_info()["diagonal_cols"] == 0
    cd = prob["cone_dims"]
    rng = np.random.default_rng(3)
    v, s = cone_point(cd, rng), cone_point(cd, rng)
    ry, rw, rv = rng.standard_normal(e1.n), rng.standard_normal(p), rng.standard_normal(e1.m)
    out = []
    for e in (e2, e1):
        lam = e.factor_from_point(v, s)
        assert e.last_factor_status == 0
        out.append([np.asarray(lam)] + [np.asarray(x) for x in e.solve(ry, rw if p else None, rv)])
    for a, b in zip(*out):
        assert np.array_equal(a, b)
    e1.close()
    e2.close()


@pytest.mark.gpu
def test_no_coupled_columns_box_qp():
    """A box QP with diagonal Q and p = 0: H is diagonal, K is empty, no Cholesky plan exists."""
    n = 500
    rng = np.random.default_rng(4)
    q = rng.uniform(0.5, 2.0, n)
    A = np.vstack([np.eye(n), -np.eye(n)])
    cd = [("R", 2 * n)]
    e = engine(dict(Q=sp.diags(q).tocsc(), A=A, G=np.zeros((0, n)), cone_dims=cd))
    assert e.split_info() == dict(enabled=1, coupled_cols=0, diagonal_cols=n, cols_from_rest=0, cols_from_Q=0,
                                  cols_from_G=0)
    v, s = cone_point(cd, rng, wide=True), cone_point(cd, rng, wide=True)
    e.nt_scaling(v, s)
    e.form_H()
    w2 = v / s                                         # (F'F)^-1 on R cones
    h = q + w2[:n] + w2[n:]
    H = e.get_H()
    assert np.array_equal(H, np.diag(np.diag(H)))
    assert np.all(np.abs(np.diag(H) - h) <= 16 * U * h)
    assert e.factor_H() == 0
    assert e.stats()["chol_flops"] == 0
    rhs = rng.standard_normal(n)
    assert np.all(np.abs(np.asarray(e.solve_H(rhs)) - rhs / h) <= 32 * U * np.abs(rhs / h))
    ry, rv = rng.standard_normal(n), rng.standard_normal(2 * n)
    dy, _, dv = e.solve(ry, None, rv)
    # Q dy - A' dv = ry,  A dy + F'F dv = rv
    K = np.block([[np.diag(q), -A.T], [A, np.diag(1.0 / w2)]])
    sol = np.linalg.solve(K, np.concatenate([ry, rv]))
    assert rel(dy, sol[:n]) < 1e-10 and rel(dv, sol[n:]) < 1e-10
    e.close()


def failing_problem(kind, n=200, p=3):
    """rho = 0.  'D': column 77 has Q_77 = 0, no bound and a G entry only: h_77 = 0 on D.  'K': Q couples 5 and 6
    with [[1, 2], [2, 1]] and neither has a bound: H_KK is indefinite at its second pivot, global column 6."""
    rng = np.random.default_rng(8)
    q = np.ones(n)
    Q = np.diag(q)
    skip = {77} if kind == "D" else {5, 6}
    if kind == "D":
        Q[77, 77] = 0.0
    else:
        Q[5, 6] = Q[6, 5] = 2.0
    A = np.array([sparse_row(n, [j], rng) for j in range(n) if j not in skip])
    G = np.zeros((p, n))
    G[:, [77, 100, 150]] = rng.standard_normal((p, 3))
    return dict(Q=Q, A=A, G=G, cone_dims=[("R", A.shape[0])])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,col", [("D", 77), ("K", 6)])
def test_pivot_failure_reports_the_global_column(kind, col):
    prob = failing_problem(kind)
    cd = prob["cone_dims"]
    rng = np.random.default_rng(9)
    v, s = cone_point(cd, rng), cone_point(cd, rng)
    rcs = []
    for mode in (2, 1):
        e = engine(prob, mode=mode, aug_rho=0.0)
        if mode == 2:
            assert (e.split_info()["diagonal_cols"] > 0)
        e.nt_scaling(v, s)
        e.form_H()
        rcs.append(e.factor_H())
        e.close()
    assert rcs == [col + 1, col + 1]


@pytest.mark.gpu
def test_solve_multi_determinism_and_mul_Q():
    prob = split_problem(seed=34)
    e, e1 = engine(prob, aug_rho=0.0), engine(prob, mode=1, aug_rho=0.0)
    assert e.split_info()["diagonal_cols"] > 0
    cd = prob["cone_dims"]
    rng = np.random.default_rng(10)
    v, s = cone_point(cd, rng), cone_point(cd, rng)
    k = 3
    RY, RW, RV = rng.standard_normal((e.n, k)), rng.standard_normal((e.p, k)), rng.standard_normal((e.m, k))
    runs = []
    for _ in range(2):
        e.factor_from_point(v, s)
        runs.append([np.asarray(x) for x in e.solve(RY[:, 0].copy(), RW[:, 0].copy(), RV[:, 0].copy())])
    for a, b in zip(*runs):
        assert np.array_equal(a, b)
    DY, DW, DV = e.solve_multi(np.asfortranarray(RY), np.asfortranarray(RW), np.asfortranarray(RV))
    for j in range(k):
        dy, dw, dv = e.solve(RY[:, j].copy(), RW[:, j].copy(), RV[:, j].copy())
        assert np.array_equal(DY[:, j], dy) and np.array_equal(DW[:, j], dw) and np.array_equal(DV[:, j], dv)
    # Q y: the same non-zero products in both modes; mode 1 sums each K row over all n columns (zeros included),
    # mode 2 over K only, so the sums are grouped differently: gamma_n |Q| |x|
    x = rng.standard_normal(e.n)
    y2, y1 = np.asarray(e.mul_Q(x)), np.asarray(e1.mul_Q(x))
    Qd = prob["Q"]
    assert np.all(np.abs(y2 - y1) <= 2 * C_H * U * (e.n + 2) * (np.abs(Qd) @ np.abs(x)))
    assert np.all(np.abs(y2 - Qd @ x) <= C_H * U * (e.n + 2) * (np.abs(Qd) @ np.abs(x)))
    e.close()
    e1.close()


@pytest.mark.gpu
@pytest.mark.parametrize("aug_rho", [-1.0, 0.0])
def test_reduced_c5_full_solve(aug_rho):
    """C5 at n = 3000, k = 16, p = 100 through cip_ipm_solve in mode 2, against mode 1 (same algorithm: status
    and iterations +-1, y / v / w to 1e-6) and against the oracle with the tolerances test_gpu_fullsize.py uses for
    this degenerate LP (iterations within 3, y to 1e-5, the objective, (v, w) through the optimality conditions)."""
    import conicip_b200 as cb
    prob = P.config5(n=3000, k=16, p=100)
    Q, c, A, b, cd, G, d = (prob[k] for k in ("Q", "c", "A", "b", "cone_dims", "G", "d"))
    e2 = cb.Engine(Q, A, G, cd, row_structure=2, aug_rho=aug_rho)
    info = e2.split_info()
    assert info == expected_split_info(Q, A, G, cd, aug_rho) and info["diagonal_cols"] > 0
    s2 = cb.conicIP_native(Q, c, A, b, cd, G, d, engine=e2, optTol=1e-8)
    e1 = cb.Engine(Q, A, G, cd, row_structure=1, aug_rho=aug_rho)
    s1 = cb.conicIP_native(Q, c, A, b, cd, G, d, engine=e1, optTol=1e-8)
    assert s2.status == s1.status == "Optimal" and abs(s2.Iter - s1.Iter) <= 1, (s2.Iter, s1.Iter)
    for f in ("y", "v", "w"):
        assert rel(getattr(s2, f), getattr(s1, f)) < 1e-6, f
    so = O.conicIP(Q, c, A, b, cd, G, d, optTol=1e-8, kktsolver=O.kktsolver_qr)
    assert so.status == "Optimal" and abs(s2.Iter - so.Iter) <= 3, (s2.Iter, so.Iter)
    assert rel(s2.y, so.y) < 1e-5
    assert abs(s2.pobj - so.pobj) <= 1e-7 * (1 + abs(so.pobj))
    assert np.linalg.norm(G.T @ s2.w - A.T @ s2.v - c) <= 1e-7 * (1 + np.linalg.norm(c))
    e1.close()
    e2.close()


@pytest.mark.gpu
def test_host_driven_conicip_matches_native():
    import conicip_b200 as cb
    prob = split_problem(seed=35)
    args = (prob["Q"], prob["c"], prob["A"], prob["b"], prob["cone_dims"], prob["G"], prob["d"])
    s_host = cb.conicIP(*args, kktsolver=cb.make_kktsolver(row_structure=2), optTol=1e-8)
    s_nat = cb.conicIP_native(*args, row_structure=2, optTol=1e-8)
    s_one = cb.conicIP_native(*args, row_structure=1, optTol=1e-8)
    assert s_host.status == s_nat.status == s_one.status == "Optimal"
    assert abs(s_host.Iter - s_nat.Iter) <= 1
    for f in ("y", "w", "v"):
        assert rel(getattr(s_host, f), getattr(s_nat, f)) < 1e-6
        assert rel(getattr(s_nat, f), getattr(s_one, f)) < 1e-6


def split_bytes_bound(n, m, p, nK, nr, nJ, max_s_order):
    """Resident bytes of a mode-2 handle, from shapes: vectors and scalings (n, m, p), G and the Schur block, the
    K block (Q_KK, rho-base, H_KK, G_K, Z_K), the rest rows (two copies over J plus their Gram matrix), the split-K
    workspace of the GEMM (2048 tiles) and the S-cone workspace, with every count rounded up generously."""
    n_pad, m_pad, p_pad, nK_pad = round_up(n), round_up(m, 32), round_up(p) if p else 0, round_up(nK)
    nr_pad, nJ_pad = round_up(nr, 32), round_up(nJ)
    doubles = (64 * (n_pad + 4) + 40 * (m_pad + 4) + 16 * (p_pad + 4)
               + 2 * p_pad * n_pad + 3 * p_pad * p_pad
               + 4 * nK_pad * nK_pad + 3 * p_pad * nK_pad + nK_pad * 128
               + 3 * nr_pad * nJ_pad + nJ_pad * nJ_pad
               + 4 * 148 * 8 * 128 + 64 * max(n, p)
               + 2048 * 128 * 128 + 2 * max_s_order ** 4)
    return 8 * doubles + (64 << 20)


@pytest.mark.gpu
def test_c5_wide_solves_at_n_150000():
    """The capability: C5 at n = 150 000 (CSC input, no Q, aug_rho = 0).  Modes 0 and 1 would hold n_pad^2 doubles
    (180 GB) per H; this handle is never created in those modes, and cip_get_H is never called."""
    import conicip_b200 as cb
    n, k, p = 150_000, 64, 1000
    prob = P.config5_sparse(n=n, k=k, p=p)
    A, G, c, b, d, cd = prob["A"], prob["G"], prob["c"], prob["b"], prob["d"], prob["cone_dims"]
    m = A.shape[0]
    e = cb.Engine(None, A, G, cd, row_structure=2, aug_rho=0.0)
    info, si = e.split_info(), e.structure_info()
    dim = k * (k + 1) // 2
    assert info == dict(enabled=1, coupled_cols=dim, diagonal_cols=n - dim, cols_from_rest=dim, cols_from_Q=0,
                        cols_from_G=0)
    y, w, v, res = e.ipm_solve(c, b, d, optTol=1e-8)
    assert res["status"] == "Optimal", res
    y, w, v = np.asarray(y), np.asarray(w), np.asarray(v)
    scale = 1 + np.linalg.norm(c)
    assert np.linalg.norm(G.T @ w - A.T @ v - c) <= 1e-7 * scale           # Q = 0
    assert np.linalg.norm(G @ y - d) <= 1e-7 * (1 + np.linalg.norm(d))
    slack = A @ y - b
    assert slack[:n].min() > -1e-7 and v[:n].min() > -1e-9
    assert np.linalg.eigvalsh(O.mat(slack[n:])).min() > -1e-7 and np.linalg.eigvalsh(O.mat(v[n:])).min() > -1e-9
    pobj, dobj = c @ y, b @ v + d @ w
    assert abs(pobj - dobj) <= 1e-6 * (1 + abs(pobj))
    st = e.stats()
    bound = split_bytes_bound(n, m, p, dim, si["rest_rows"], si["rest_cols"], k)
    assert st["device_bytes"] <= bound, (st["device_bytes"], bound)
    assert st["device_bytes"] < 8 * round_up(n) ** 2 / 50
    e.close()


@pytest.mark.gpu
def test_sharded_handle_is_rejected():
    import conicip_b200 as cb
    prob = P.box_qp(64)
    for A in (prob["A"], sp.csc_matrix(prob["A"])):
        with pytest.raises(cb.CipError, match="single-device"):
            cb.Engine(prob["Q"], A, None, prob["cone_dims"], ngpus=2, row_structure=2)
