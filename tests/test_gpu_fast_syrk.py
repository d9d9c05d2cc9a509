"""The fast SYRK of form_H (csrc/fast_syrk.cu): a blocked SYRK whose off-diagonal blocks take one Strassen-Winograd
level on columns equilibrated by powers of two.

The library takes it by itself only at large n; CIP_FAST_SYRK=1 forces it on any dense single-device handle whose
rows are all R rows (and CIP_FAST_SYRK_LEAF sets the width of the diagonal blocks), so these tests reach it at
n ~ 1000.  H is checked against a reference more accurate than FP64 (np.longdouble) with the metric
max |dH_ij| / sqrt(H_ii H_jj), the error form a Cholesky factorisation is invariant to.
"""
import numpy as np
import pytest

import oracle as O

U = 2.0 ** -53

# err(H) <= C_FAST * u * m.  One Winograd level adds one rounding per operand sum on each side (3 levels of sums
# at most), one per product combination (4 adds) and the unscaling (exact): with columns equilibrated to within a
# factor of 2 each sum is bounded by ~4 column norms, so the product error is at most ~16 gamma_{m/2} plus a few u.
# The classical SYRK is within gamma_m.  A wrong sign, a misplaced block, Q added twice or unequilibrated columns
# of very different norms miss this by many orders of magnitude.
C_FAST = 16
# the fast path against the classical one on the same input (both against the same reference)
RATIO = 16


@pytest.fixture(autouse=True)
def _no_knobs(monkeypatch):
    for k in ("CIP_FAST_SYRK", "CIP_FAST_SYRK_LEAF", "CIP_FOLD_SCALING", "CIP_ROW_STRUCTURE"):
        monkeypatch.delenv(k, raising=False)


def problem(n, m, seed, col_exp=0):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    if col_exp:
        A *= np.exp2(rng.integers(-col_exp, col_exp + 1, n))[None, :]
    B = rng.standard_normal((n, 8)) / np.sqrt(8)
    Q = B @ B.T + np.diag(1.0 + rng.uniform(size=n))
    return Q, A


def scaling(m, seed, wide):
    rng = np.random.default_rng(seed + 1)
    # F = diag(sqrt(s / v)): central s/v in [0.25, 4], wide from 1e-8 to 1e8
    lo, hi = (-8.0, 8.0) if wide else (-0.6, 0.6)
    return np.sqrt(10.0 ** rng.uniform(lo, hi, m))


def engine(monkeypatch, Q, A, fast, leaf=None, **kw):
    import conicip_b200 as cb
    monkeypatch.setenv("CIP_FAST_SYRK", "1" if fast else "0")
    if leaf:
        monkeypatch.setenv("CIP_FAST_SYRK_LEAF", str(leaf))
    else:
        monkeypatch.delenv("CIP_FAST_SYRK_LEAF", raising=False)
    return cb.Engine(Q, A, None, [("R", A.shape[0])], **kw)


def form(eng, d):
    import conicip_b200 as cb
    eng.set_scaling(cb.Block([cb.Diagonal(d)]))
    eng.form_H()
    return np.tril(eng.get_H())


def ref_H(Q, A, d):
    X = (A / d[:, None]).astype(np.longdouble)      # Atil = F^-T A, as the device rounds it (one product per entry)
    return np.tril(Q.astype(np.longdouble) + X.T @ X)


def err(H, R):
    dg = np.sqrt(np.diag(R).astype(np.float64))
    return float(np.max(np.abs((H.astype(np.longdouble) - R).astype(np.float64)) / np.outer(dg, dg)))


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [False, True], ids=["central", "wide"])
@pytest.mark.parametrize("col_exp", [0, 40], ids=["plain", "cols2^40"])
@pytest.mark.parametrize("n,m,leaf", [(512, 1030, None), (1000, 1030, 256)], ids=["depth1", "depth2_ragged"])
def test_fast_H_against_extended_precision(monkeypatch, n, m, leaf, col_exp, wide):
    """H = Q + Atil'Atil of the fast path (and of the classical path) against a long-double reference, at a
    central and a wide NT scaling, with columns of A scaled by up to 2^+-40 (which equilibration has to absorb)."""
    Q, A = problem(n, m, seed=n + col_exp, col_exp=col_exp)
    d = scaling(m, n, wide)
    R = ref_H(Q, A, d)
    ef = err(form(engine(monkeypatch, Q, A, True, leaf), d), R)
    ec = err(form(engine(monkeypatch, Q, A, False), d), R)
    print(f"n={n} m={m} leaf={leaf} cols=2^+-{col_exp} wide={wide}: fast {ef / U:.1f} u, classical {ec / U:.1f} u")
    assert ef <= C_FAST * U * m
    assert ef <= RATIO * max(ec, U)


@pytest.mark.gpu
def test_fast_path_runs_and_classical_is_untouched(monkeypatch):
    """Forced on, the product differs from the classical SYRK in the last bits (the fast path ran); automatic at
    small n, and forced on a folded or row-structured handle, H is bit-identical to the classical path."""
    n, m = 512, 1024
    Q, A = problem(n, m, seed=3)
    d = scaling(m, 3, False)
    H0 = form(engine(monkeypatch, Q, A, False), d)
    Hf = form(engine(monkeypatch, Q, A, True), d)
    assert not np.array_equal(Hf, H0)
    monkeypatch.delenv("CIP_FAST_SYRK", raising=False)
    import conicip_b200 as cb
    assert np.array_equal(form(cb.Engine(Q, A, None, [("R", m)]), d), H0)       # below the size threshold
    for kw in (dict(fold_scaling=1), dict(row_structure=1)):
        H0k = form(engine(monkeypatch, Q, A, False, **kw), d)
        assert np.array_equal(form(engine(monkeypatch, Q, A, True, **kw), d), H0k), kw


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [None, 256])
def test_fast_cholesky_and_solve(monkeypatch, leaf):
    """Cholesky and a KKT solve on the fast H against the oracle, with the tolerances of the classical path's test
    (test_gpu_kernels.py::test_form_H_cholesky_and_solve)."""
    n, m = 1000, 3030
    Q, A = problem(n, m, seed=11)
    rng = np.random.default_rng(5)
    v, s = rng.uniform(0.5, 1.5, m), rng.uniform(0.5, 1.5, m)
    cd = [("R", m)]
    eng = engine(monkeypatch, Q, A, True, leaf)
    eng.nt_scaling(v, s)
    Fo = O.Block([O.Diag(np.sqrt(s / v))])
    At = Fo.inv_adjoint().mul(A)
    Href = Q + At.T @ At
    rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))
    eng.form_H()
    assert rel(np.tril(eng.get_H()), np.tril(Href)) < 1e-12
    assert eng.factor_H() == 0
    assert rel(np.tril(eng.get_H()), np.linalg.cholesky(Href)) < 1e-11
    ry, rv = rng.standard_normal(n), rng.standard_normal(m)
    dy, _, dv = eng.solve(ry, None, rv)
    G = np.zeros((0, n))
    for ks in (O.kktsolver_chol, O.pivot(O.kktsolver_2x2), O.kktsolver_qr):
        oy, _, ov = ks(Q, A, G, cd)(Fo, Fo.inv_adjoint())(ry, np.zeros(0), rv)
        assert rel(dy, oy) < 1e-9 and rel(dv, ov) < 1e-9


@pytest.mark.gpu
def test_fast_ipm_solve_c2_shape(monkeypatch):
    """The native interior-point loop on a C2-shaped problem (dense QP, m = 2n R rows) with the fast path forced:
    the same status as the classical path, iterations within one, and a converged solution."""
    from conicip_b200 import problems as P
    pr = P.config2(n=2048, m=4096, seed=2)
    out = {}
    for fast in (False, True):
        eng = engine(monkeypatch, pr["Q"], pr["A"], fast)
        y, w, v, info = eng.ipm_solve(pr["c"], pr["b"], optTol=1e-8)
        out[fast] = (info, y)
        eng.close()
    (ic, yc), (i_f, yf) = out[False], out[True]
    assert i_f["status"] == ic["status"] == "Optimal"
    assert abs(i_f["Iter"] - ic["Iter"]) <= 1
    assert max(i_f["prFeas"], i_f["duFeas"], i_f["muFeas"]) < 1e-8
    assert np.linalg.norm(np.asarray(yf) - np.asarray(yc)) <= 1e-6 * np.linalg.norm(np.asarray(yc))
