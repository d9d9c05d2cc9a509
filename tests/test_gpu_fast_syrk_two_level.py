"""The second Winograd level of the fast SYRK (csrc/fast_syrk.cu): where the off-diagonal blocks are wide, each of
their seven products is itself done as seven products of half size.

The library takes the second level by itself only where the level-2 products are at least 1024 columns wide (n of
12288 and more); CIP_FAST_SYRK_LEVELS=2 forces it on every depth whose level-2 products split into whole 128-tiles,
so these tests reach it at n ~ 1000-2000.  H is checked against a long-double reference with the metric
max |dH_ij| / sqrt(H_ii H_jj), as in test_gpu_fast_syrk.py.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

U = 2.0 ** -53
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# err(H) <= C_TWO * u * m.  The one-level bound C_FAST = 16 (test_gpu_fast_syrk.py) counts operand sums of up to 4
# equilibrated columns on each side of a product.  The second level sums blocks of those operands once more, so an
# operand of a level-2 product is a signed sum of up to 4 level-1 operands: its norm, and so the error of its
# product, grows by up to another 4 on each side, while the contraction halves (gamma_{m/4} instead of gamma_{m/2}).
# That gives 16 * 16 / 2 = 128 for the products; the two combinations add a few u.  A wrong sign, a tile written
# off its place, a product unscaled twice, a wrong contraction half or unequilibrated sums of columns scaled by
# 2^+-40 miss this by many orders of magnitude.
# This absolute bound is a worst case, so it is loose (1.3e5 u at m = 1030): it catches those O(1) defects, not a
# loss of accuracy by a factor of 100.  RATIO is the real accuracy guard.
C_TWO = 128
# two levels against one level on the same input (both against the same reference): one more level of sums, up to
# 4 x 4 on the operand norms of the product it is applied to.  This bounds what the second level may add.
RATIO = 16

KNOBS = ("CIP_FAST_SYRK", "CIP_FAST_SYRK_LEAF", "CIP_FAST_SYRK_LEVELS", "CIP_FOLD_SCALING", "CIP_ROW_STRUCTURE")


@pytest.fixture(autouse=True)
def _no_knobs(monkeypatch):
    for k in KNOBS:
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
    lo, hi = (-8.0, 8.0) if wide else (-0.6, 0.6)
    return np.sqrt(10.0 ** rng.uniform(lo, hi, m))


def engine(monkeypatch, Q, A, fast, levels=None, leaf=None, **kw):
    """fast: CIP_FAST_SYRK=1 (else 0); levels: CIP_FAST_SYRK_LEVELS (None: the library's rule)."""
    import conicip_b200 as cb
    monkeypatch.setenv("CIP_FAST_SYRK", "1" if fast else "0")
    for k, v in (("CIP_FAST_SYRK_LEVELS", levels), ("CIP_FAST_SYRK_LEAF", leaf)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))
    return cb.Engine(Q, A, None, [("R", A.shape[0])], **kw)


def form(eng, d):
    import conicip_b200 as cb
    eng.set_scaling(cb.Block([cb.Diagonal(d)]))
    eng.form_H()
    H = np.tril(eng.get_H())
    eng.close()
    return H


def ref_H(Q, A, d):
    X = (A / d[:, None]).astype(np.longdouble)
    return np.tril(Q.astype(np.longdouble) + X.T @ X)


def err(H, R):
    dg = np.sqrt(np.diag(R).astype(np.float64))
    return float(np.max(np.abs((H.astype(np.longdouble) - R).astype(np.float64)) / np.outer(dg, dg)))


# n = 1024: one depth, at two levels.  n = 2000 (padded to 2048, ragged), leaf 256: depths 0 and 1 at two levels
# (level-2 products 256 and 128 wide), depth 2 at one (64 is not a whole tile).
SHAPES = [(1024, 1030, None), (2000, 1030, 256)]
SHAPE_IDS = ["depth0_two", "mixed_ragged"]


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [False, True], ids=["central", "wide"])
@pytest.mark.parametrize("col_exp", [0, 40], ids=["plain", "cols2^40"])
@pytest.mark.parametrize("n,m,leaf", SHAPES, ids=SHAPE_IDS)
def test_two_level_H_against_extended_precision(monkeypatch, n, m, leaf, col_exp, wide):
    """H of the two-level path against a long-double reference, at a central and a wide NT scaling, with columns of
    A scaled by up to 2^+-40; and against the error of the one-level path on the same input."""
    Q, A = problem(n, m, seed=n + col_exp, col_exp=col_exp)
    d = scaling(m, n, wide)
    R = ref_H(Q, A, d)
    e2 = err(form(engine(monkeypatch, Q, A, True, 2, leaf), d), R)
    e1 = err(form(engine(monkeypatch, Q, A, True, 1, leaf), d), R)
    print(f"n={n} m={m} leaf={leaf} cols=2^+-{col_exp} wide={wide}: two levels {e2 / U:.1f} u, one {e1 / U:.1f} u")
    assert e2 <= C_TWO * U * m
    assert e2 <= RATIO * max(e1, U)


@pytest.mark.gpu
def test_two_level_path_runs_and_nothing_else_changes(monkeypatch):
    """Forced, the second level changes H in the last bits (it ran); the library's own choice at these sizes is one
    level, bit for bit; folded and row-structured handles ignore the knob."""
    n, m, leaf = 2000, 1030, 256
    Q, A = problem(n, m, seed=7)
    d = scaling(m, 7, False)
    H1 = form(engine(monkeypatch, Q, A, True, 1, leaf), d)
    H2 = form(engine(monkeypatch, Q, A, True, 2, leaf), d)
    assert not np.array_equal(H2, H1)
    assert np.array_equal(form(engine(monkeypatch, Q, A, True, None, leaf), d), H1)
    for kw in (dict(fold_scaling=1), dict(row_structure=1)):
        H0k = form(engine(monkeypatch, Q, A, True, 1, leaf, **kw), d)
        assert np.array_equal(form(engine(monkeypatch, Q, A, True, 2, leaf, **kw), d), H0k), kw


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [None, 256], ids=["depth0_two", "mixed"])
def test_two_level_cholesky_and_solve(monkeypatch, leaf):
    """Cholesky and a KKT solve on the two-level H against the oracle, with the tolerances of
    test_gpu_fast_syrk.py::test_fast_cholesky_and_solve."""
    n, m = 1000, 3030
    Q, A = problem(n, m, seed=11)
    rng = np.random.default_rng(5)
    v, s = rng.uniform(0.5, 1.5, m), rng.uniform(0.5, 1.5, m)
    cd = [("R", m)]
    eng = engine(monkeypatch, Q, A, True, 2, leaf)
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
    eng.close()


@pytest.mark.gpu
def test_two_level_ipm_solve_c2_shape(monkeypatch):
    """The native interior-point loop on a C2-shaped problem with two levels forced: Optimal like the classical
    path, iterations within one, and a converged solution."""
    from conicip_b200 import problems as P
    pr = P.config2(n=2048, m=4096, seed=2)
    out = {}
    for fast in (False, True):
        eng = engine(monkeypatch, pr["Q"], pr["A"], fast, 2 if fast else None)
        y, w, v, info = eng.ipm_solve(pr["c"], pr["b"], optTol=1e-8)
        out[fast] = (info, y)
        eng.close()
    (ic, yc), (i_f, yf) = out[False], out[True]
    assert i_f["status"] == ic["status"] == "Optimal"
    assert abs(i_f["Iter"] - ic["Iter"]) <= 1
    assert max(i_f["prFeas"], i_f["duFeas"], i_f["muFeas"]) < 1e-8
    assert np.linalg.norm(np.asarray(yf) - np.asarray(yc)) <= 1e-6 * np.linalg.norm(np.asarray(yc))


def test_timing_script_classifies_phases_by_kernel_name():
    """scripts/fast_syrk_timing.py attributes gemm launches to the combination that reads them (no device)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "fast_syrk_timing.py"), "--selftest"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "selftest ok" in r.stdout
