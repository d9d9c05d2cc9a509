"""`cip_options.row_structure = 1` against an independent FP64 evaluation of H, A and the KKT solve.

tests/test_gpu_row_structure.py compares the structured handle with the same library with the option off.  Here
the reference is computed on the host from the oracle's scaling blocks, H is compared element by element against
a rounding-error bound, and the problems are shaped to reach the branches of csrc/structure.cu a comparison with
the off path cannot discriminate: a compressed column set J that is not the identity, a folded rest whose order
is not the global row order, rest cones renumbered around dropped R cones, the compression threshold itself, a
rest that touches no column, host-supplied scalings, Julia-style CSC input and ragged or very tall shapes.

The first part (the reference, the comparator and the mirror of the classification rule) runs without a GPU.
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
from conicip_b200 import problems as P

U = 2.0 ** -53          # unit roundoff of float64
TILE = 128              # H is stored in 128 x 128 tiles; J is padded to a multiple of it

# C_H: |H_dev - H_ref| <= C_H * u * (k + 2) * B elementwise.  A sum of k products, in any order, is within
# gamma_k * sum |x_i y_i| of the exact value (gamma_k = k u / (1 - k u), Higham, Accuracy and Stability, sec. 3.1).
# The device and the reference each make that error once for the contraction over the rows (k counts every row of
# A and G) and once more in each factor of F^-T A (at most the largest cone, also counted in k); their scalings are
# computed independently from the same (v, s) and differ by a few ulps per entry.  That is at most 2 * 2 gamma_k
# plus a few u in all: C_H = 4 with the "+ 2".  A wrong entry of H is wrong by a sizeable fraction of B, far
# beyond this bound.
C_H = 4


@pytest.fixture(autouse=True)
def _option_decides(monkeypatch):
    # CIP_ROW_STRUCTURE=1 would turn a handle created with row_structure=0 structured as well
    monkeypatch.delenv("CIP_ROW_STRUCTURE", raising=False)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def round_up(x, t=TILE):
    return (x + t - 1) // t * t


def dense(M, shape):
    if M is None:
        return np.zeros(shape)
    return M.toarray() if sp.issparse(M) else np.asarray(M, dtype=np.float64)


# ================================================================ reference, bound, mirror
def oracle_F(cone_dims, v, s):
    """The NT scaling of (v, s) from the oracle's own formulas (not the engine's get_scaling)."""
    bl, off = [], 0
    for t, k in cone_dims:
        xv, xs = v[off:off + k], s[off:off + k]
        bl.append(O.Diag(np.sqrt(xs / xv)) if t == "R" else O.nestod_soc(xv, xs) if t == "Q" else O.nestod_sdc(xv, xs))
        off += k
    return O.Block(bl)


def ref_H(Q, A, G, cone_dims, F, rho, delta=0.0):
    """H = Q + (F^-T A)'(F^-T A) + rho G'G + delta I in float64, with the bound matrix
    B = |Q| + (|F^-T| |A|)'(|F^-T| |A|) + rho |G|'|G| + |delta| I and the contraction length k."""
    A = dense(A, None)
    m, n = A.shape
    Qd = dense(Q, (n, n))
    Gd = dense(G, (0, n))
    At, Ab = np.empty_like(A), np.empty_like(A)
    off, kc = 0, 1
    for i, (t, k) in enumerate(cone_dims):
        Fit = F[i].inv().adjoint()
        Ai = A[off:off + k]
        if isinstance(Fit, O.Diag):
            At[off:off + k] = Fit.diag[:, None] * Ai
            Ab[off:off + k] = np.abs(Fit.diag)[:, None] * np.abs(Ai)
        else:
            D = Fit.dense()
            At[off:off + k] = D @ Ai
            Ab[off:off + k] = np.abs(D) @ np.abs(Ai)
            kc = max(kc, k)
        off += k
    H = Qd + At.T @ At + rho * (Gd.T @ Gd) + delta * np.eye(n)
    B = np.abs(Qd) + Ab.T @ Ab + rho * (np.abs(Gd).T @ np.abs(Gd)) + abs(delta) * np.eye(n)
    return SimpleNamespace(H=H, B=B, k=m + Gd.shape[0] + kc)


def H_violations(H, ref):
    """Lower-triangle entries of H outside the rounding-error bound of the reference (NaN counts as outside)."""
    tol = C_H * U * (ref.k + 2) * ref.B
    return np.tril(~(np.abs(H - ref.H) <= tol)), tol


def assert_H(H, ref, what=""):
    bad, tol = H_violations(H, ref)
    if bad.any():
        i, j = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {int(bad.sum())} entries of H outside the bound, first H[{i},{j}] = "
                             f"{H[i, j]!r}, reference {ref.H[i, j]!r}, bound {tol[i, j]:.3e}")


def assert_diag_tiles_symmetric(H, ref, what=""):
    """Inside each 128 x 128 diagonal tile the device keeps both halves of H (structure.cu, scatter_gram_kernel)."""
    tol = C_H * U * (ref.k + 2) * ref.B
    n = H.shape[0]
    for t0 in range(0, n, TILE):
        s = slice(t0, min(n, t0 + TILE))
        T, Tt = H[s, s], tol[s, s]
        bad = ~(np.abs(T - T.T) <= Tt)
        assert not bad.any(), f"{what}: diagonal tile at {t0} is not symmetric at {np.argwhere(bad)[0] + t0}"


def assert_matvec(got, A, x, what=""):
    """Elementwise: |A x - got| <= C_H u (k + 2) (|A| |x|) with k the length of the contraction."""
    want = A @ x
    bound = C_H * U * (A.shape[1] + 2) * (np.abs(A) @ np.abs(x))
    bad = ~(np.abs(np.asarray(got) - want) <= bound)
    assert not bad.any(), f"{what}: entry {np.argwhere(bad)[0]} of the product outside the bound"


def expected_structure_info(A, cone_dims, n, p, aug_rho=-1.0):
    """The classification rule of row_structure = 1, restated: an R row with exactly one non-zero (a value
    != 0.0, so -0.0 is zero) is a singleton, an R row without one is empty, every other row (all Q and S rows, R
    rows with two or more non-zeros) is in the rest.  J = the columns the rest touches; the rest is compressed onto
    J when roundup(|J|, 128) <= roundup(n, 128) / 2.  Q + rho G'G is the constant base when p > 0 and rho > 0
    (rho = 1 by default when p > 0)."""
    A = dense(A, None)
    m = A.shape[0]
    if m == 0:
        return dict(enabled=0, singleton_rows=0, empty_rows=0, rest_rows=0, rest_cols=0, compressed=0,
                    base_has_gtg=0)
    nz = A != 0.0
    cnt = nz.sum(axis=1)
    is_r = np.concatenate([np.full(k, t == "R") for t, k in cone_dims])
    sing = is_r & (cnt == 1)
    empty = is_r & (cnt == 0)
    rest = ~(sing | empty)
    nr = int(rest.sum())
    nJ = int(nz[rest].any(axis=0).sum())
    compressed = nr > 0 and round_up(nJ) <= round_up(n) // 2
    rho = aug_rho if aug_rho >= 0 else (1.0 if p > 0 else 0.0)
    return dict(enabled=1, singleton_rows=int(sing.sum()), empty_rows=int(empty.sum()), rest_rows=nr,
                rest_cols=nJ if compressed else (n if nr > 0 else 0), compressed=int(compressed),
                base_has_gtg=int(p > 0 and rho > 0))


# ================================================================ problems
def cone_point(cone_dims, rng, wide=False):
    """A strictly interior point of the cone product.  wide: R entries spread over 1e-4 .. 1e4 and every Q / S
    block scaled by one factor in that range, so v / s spans 1e-8 .. 1e8 as near convergence."""
    x = []
    for t, k in cone_dims:
        if t == "R":
            x.append(10.0 ** rng.uniform(-4, 4, k) if wide else rng.uniform(0.5, 1.5, k))
            continue
        if t == "Q":
            u = 0.2 * rng.standard_normal(k - 1)
            blk = np.concatenate([[1.0 + np.linalg.norm(u)], u])
        else:
            o = O.ord_(k)
            B = rng.standard_normal((o, o)) / np.sqrt(o)
            blk = O.vecm(B @ B.T + np.eye(o))
        x.append(blk * (10.0 ** rng.uniform(-4, 4) if wide else 1.0))
    return np.concatenate(x)


def sparse_row(n, cols, rng):
    a = np.zeros(n)
    a[cols] = rng.choice([-1.0, 1.0], len(cols)) * rng.uniform(0.5, 2.0, len(cols))
    return a


def rest_row(n, J, r, rng, extra):
    """Row r of a family that covers J: columns J[2r], J[2r + 1] (cyclically) and `extra` more from J."""
    cols = np.concatenate([J[[2 * r % len(J), (2 * r + 1) % len(J)]], rng.choice(J, extra, replace=False)])
    return sparse_row(n, np.unique(cols), rng)


def finish(name, A, cone_dims, p, rng, Q=None):
    """Strictly feasible (b = A y0 - s0, d = G y0, s0 interior) with Q positive definite: bounded."""
    A = np.array(A, dtype=np.float64)
    n = A.shape[1]
    y0 = rng.standard_normal(n)
    b = A @ y0 - cone_point(cone_dims, rng)
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    Q = P._lowrank_q(rng, n, 8) if Q is None else Q
    return P._prob(name, Q, rng.standard_normal(n), A, b, cone_dims, G, G @ y0, optTol=1e-8)


def scattered_problem(seed=21, n=1000, p=5):
    """A bound on every column (singletons) interleaved with rest rows over ~150 scattered columns J: 0, n-1 and
    columns of every 128-tile; one rest row spans 0 and n-1; a Q cone of rest rows sits between two R cones."""
    rng = np.random.default_rng(seed)
    J = np.sort(np.concatenate([[0, n - 1], rng.choice(np.arange(1, n - 1), 148, replace=False)]))
    assert len(set(J // TILE)) >= 3
    rows, r = [sparse_row(n, [0, n - 1, J[len(J) // 2]], rng)], 0
    for t, j in enumerate(rng.permutation(n)):
        rows.append(sparse_row(n, [j], rng))
        if t % 5 == 0:
            rows.append(rest_row(n, J, r, rng, rng.integers(0, 5)))
            r += 1
    cones = [("R", len(rows))]
    rows += [sparse_row(n, rng.choice(J, 8, replace=False), rng) / 4 for _ in range(6)]
    cones.append(("Q", 6))
    rows += [sparse_row(n, rng.choice(J, 3, replace=False), rng) for _ in range(40)]
    cones.append(("R", 40))
    return finish("scattered_J", np.array(rows), cones, p, rng)


def folded_problem(seed=22, n=600, p=3):
    """R cones only (the rest folds): singletons and empty rows before and between rest rows over ~150 of n
    columns, so rest order differs from global order and the rest is compressed."""
    rng = np.random.default_rng(seed)
    J = np.sort(rng.choice(n, 150, replace=False))
    rows, r, t = [], 0, 0
    sing = list(rng.permutation(n))
    while sing:
        kind = "SSRSERS"[t % 7]                  # singleton, rest, empty
        t += 1
        if kind == "S":
            rows.append(sparse_row(n, [sing.pop()], rng))
        elif kind == "E":
            rows.append(np.zeros(n))
        else:
            rows.append(rest_row(n, J, r, rng, rng.integers(0, 4)))
            r += 1
    rows = np.array(rows)
    half = len(rows) // 2
    return finish("folded_rest", rows, [("R", half), ("R", len(rows) - half)], p, rng)


def remap_problem(seed=23, n=80, p=4):
    """Cones R (all singletons), Q, R (0 / 1 / 2+ non-zeros), S of order 5, R (all empty), Q, and equalities: the
    rest cones are renumbered around the two dropped R cones."""
    rng = np.random.default_rng(seed)
    cols = rng.permutation(n)
    blocks = [np.array([sparse_row(n, [j], rng) for j in cols[:40]])]
    blocks.append(rng.standard_normal((5, n)) / np.sqrt(n))
    mixed = []
    for t in range(30):
        kd = t % 3
        mixed.append(np.zeros(n) if kd == 0 else sparse_row(n, rng.choice(n, 1 if kd == 1 else 5, replace=False), rng))
    blocks.append(np.array(mixed))
    blocks.append(rng.standard_normal((15, n)) / np.sqrt(n))
    blocks.append(np.zeros((8, n)))
    blocks.append(rng.standard_normal((4, n)) / np.sqrt(n))
    cones = [("R", 40), ("Q", 5), ("R", 30), ("S", 15), ("R", 8), ("Q", 4)]
    return finish("cone_remap", np.vstack(blocks), cones, p, rng)


def threshold_problem(nJ, seed=24, n=1000, p=2):
    """A bound on every column and rest rows that touch exactly nJ columns."""
    rng = np.random.default_rng(seed)
    J = rng.permutation(n)[:nJ]
    rows = [sparse_row(n, [j], rng) for j in range(n)]
    for t in range(0, nJ, 3):             # every third column of J starts a rest row, between the bounds
        rows.insert(t // 3 * 7 + 1, sparse_row(n, np.unique(np.concatenate([J[t:t + 3], rng.choice(J, 1)])), rng))
    A = np.array(rows)
    assert np.count_nonzero(A[np.count_nonzero(A, axis=1) >= 2].any(axis=0)) == nJ
    return finish("threshold", A, [("R", len(rows))], p, rng)


def empty_J_problem(seed=25, n=200, p=3):
    """Bounds as singletons plus a Q cone and an S cone whose rows of A are all zero (constant cone constraints):
    the rest has rows but touches no column."""
    rng = np.random.default_rng(seed)
    A = np.vstack([np.diag(rng.uniform(0.5, 2.0, n)), np.zeros((4 + 3, n))])
    return finish("empty_J", A, [("R", n), ("Q", 4), ("S", 3)], p, rng)


# ================================================================ device helpers
def engine(prob, A=None, Q="prob", **kw):
    import conicip_b200 as cb
    G = prob["G"] if prob["G"].shape[0] else None
    return cb.Engine(prob["Q"] if isinstance(Q, str) else Q, prob["A"] if A is None else A, G, prob["cone_dims"],
                     row_structure=1, **kw)


def rho_of(prob, aug_rho=-1.0):
    p = prob["G"].shape[0]
    return (aug_rho if aug_rho >= 0 else 1.0) if p > 0 else 0.0


def check_info(e, prob, aug_rho=-1.0):
    want = expected_structure_info(prob["A"], prob["cone_dims"], len(prob["c"]), prob["G"].shape[0], aug_rho)
    assert e.structure_info() == want
    return want


def check_H_at(e, prob, v, s, Q="prob", aug_rho=-1.0, delta=0.0, what=""):
    """form H at the NT scaling of (v, s) and compare it with the reference; returns (oracle F, reference)"""
    e.nt_scaling(v, s)
    e.form_H()
    H = e.get_H()
    Fo = oracle_F(prob["cone_dims"], v, s)
    ref = ref_H(prob["Q"] if isinstance(Q, str) else Q, prob["A"], prob["G"], prob["cone_dims"], Fo,
                rho_of(prob, aug_rho), delta)
    assert_H(H, ref, what)
    assert_diag_tiles_symmetric(H, ref, what)
    return Fo, ref


def check_H_two_points(e, prob, seed, **kw):
    rng = np.random.default_rng(seed)
    out = None
    for wide in (True, False):            # the well-conditioned point last: the handle keeps its scaling
        cd = prob["cone_dims"]
        v, s = cone_point(cd, rng, wide), cone_point(cd, rng, wide)
        out = check_H_at(e, prob, v, s, what="wide" if wide else "central", **kw)
    return out


def oracle_kkt(prob):
    return O.kktsolver_qr if any(t == "S" for t, _ in prob["cone_dims"]) else O.pivot(O.kktsolver_2x2)


def check_solve(e, prob, Fo, ref, rng, Q="prob"):
    """factor the resident H, solve one right-hand side, compare with the oracle and check the 3x3 system"""
    Qd = dense(prob["Q"] if isinstance(Q, str) else Q, (len(prob["c"]),) * 2)
    A, G, cd = prob["A"], prob["G"], prob["cone_dims"]
    n, m, p = A.shape[1], A.shape[0], G.shape[0]
    assert e.factor_H() == 0
    ry, rw, rv = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(m)
    dy, dw, dv = e.solve(ry, rw if p else None, rv)
    oy, ow, ov = oracle_kkt(prob)(Qd, A, G, cd)(Fo, Fo.inv_adjoint())(ry, rw, rv)
    assert rel(dy, oy) < 1e-9 and rel(dv, ov) < 1e-9
    if p:
        assert rel(dw, ow) < 1e-8
    Fd = Fo.dense()
    FtF = Fd.T @ Fd
    scale = np.linalg.norm(np.concatenate([ry, rw, rv]))
    assert np.linalg.norm(Qd @ dy + (G.T @ dw if p else 0) - A.T @ dv - ry) < 1e-10 * scale * (1 + np.linalg.norm(ref.H))
    assert np.linalg.norm(A @ dy + FtF @ dv - rv) < 1e-10 * scale * (1 + np.linalg.norm(FtF))
    if p:
        assert np.linalg.norm(G @ dy - rw) < 1e-10 * scale
    return dy, dw, dv


def check_matvecs(e, A, seed):
    rng = np.random.default_rng(seed)
    x, u = rng.standard_normal(A.shape[1]), rng.standard_normal(A.shape[0])
    assert_matvec(e.mul_A(x), A, x, "A x")
    assert_matvec(e.mul_A(u, trans=True), A.T, u, "A' u")
    return x, u


def check_solve_multi(e, rng):
    k = 3
    RY, RW, RV = rng.standard_normal((e.n, k)), rng.standard_normal((e.p, k)), rng.standard_normal((e.m, k))
    DY, DW, DV = e.solve_multi(np.asfortranarray(RY), np.asfortranarray(RW) if e.p else None, np.asfortranarray(RV))
    for j in range(k):
        dy, dw, dv = e.solve(RY[:, j].copy(), RW[:, j].copy() if e.p else None, RV[:, j].copy())
        assert np.array_equal(DY[:, j], dy) and np.array_equal(DV[:, j], dv)
        assert e.p == 0 or np.array_equal(DW[:, j], dw)


def full_case(prob, seed, **kw):
    """structure_info, H at two scalings (with the tile symmetry), A x, A'u, one solve, solve_multi"""
    e = engine(prob, **kw)
    info = check_info(e, prob)
    Fo, ref = check_H_two_points(e, prob, seed)
    check_matvecs(e, prob["A"], seed + 1)
    rng = np.random.default_rng(seed + 2)
    check_solve(e, prob, Fo, ref, rng)
    check_solve_multi(e, rng)
    e.close()
    return info


# ================================================================ 1. CPU: the comparator and the mirror
def test_comparator_accepts_reference_and_rejects_wrong_terms():
    prob = scattered_problem()
    A, cd = prob["A"], prob["cone_dims"]
    rng = np.random.default_rng(0)
    v, s = cone_point(cd, rng), cone_point(cd, rng)
    F = oracle_F(cd, v, s)
    ref = ref_H(prob["Q"], A, prob["G"], cd, F, 1.0)
    assert not H_violations(ref.H, ref)[0].any()
    # the same H with the cones summed in the opposite order is inside the bound too
    off = np.concatenate([[0], np.cumsum([k for _, k in cd])])
    back = np.vstack([A[off[i]:off[i + 1]] for i in reversed(range(len(cd)))])
    flip = ref_H(prob["Q"], back, prob["G"], cd[::-1], O.Block([F[i] for i in reversed(range(len(cd)))]), 1.0)
    assert not H_violations(flip.H, ref)[0].any()
    assert not np.array_equal(flip.H, ref.H)

    cnt = np.count_nonzero(A, axis=1)
    r_rows = np.arange(cd[0][1])
    # (a) one singleton term missing from the diagonal
    i = r_rows[cnt[r_rows] == 1][7]
    j = int(np.flatnonzero(A[i])[0])
    H = ref.H.copy()
    H[j, j] -= (A[i, j] / F[0].diag[i]) ** 2
    assert H_violations(H, ref)[0][j, j]
    # (b) the rest's contribution to one off-diagonal pair of J landing in the neighbouring column
    rest = ~((cnt <= 1) & np.concatenate([np.full(k, t == "R") for t, k in cd]))
    Hr = ref_H(None, A * rest[:, None], None, cd, F, 0.0).H
    J = np.flatnonzero(np.abs(A[rest]).sum(axis=0))
    pairs = [(a, b) for a in J for b in J if a > b + 1 and Hr[a, b] != 0 and Hr[a, b + 1] == 0]
    a, b = pairs[len(pairs) // 2]
    H = ref.H.copy()
    H[a, b] -= Hr[a, b]
    H[a, b + 1] += Hr[a, b]
    bad = H_violations(H, ref)[0]
    assert bad[a, b] and bad[a, b + 1]
    # (c) one rest row of an R cone scaled with another row's w
    i, i2 = r_rows[cnt[r_rows] >= 2][:2]
    d = F[0].diag.copy()
    d[i] = d[i2] * 1.5 if d[i] == d[i2] else d[i2]
    Fm = O.Block([O.Diag(d)] + [F[c] for c in range(1, len(cd))])
    assert H_violations(ref_H(prob["Q"], A, prob["G"], cd, Fm, 1.0).H, ref)[0].any()


def test_structure_info_mirror_reproduces_known_splits():
    from test_gpu_row_structure import mixed_problem
    prob = mixed_problem()
    info = expected_structure_info(prob["A"], prob["cone_dims"], 120, 7)
    assert (info["singleton_rows"], info["empty_rows"], info["rest_rows"]) == (30, 10, 35)
    assert info["compressed"] == 0 and info["rest_cols"] == 120 and info["base_has_gtg"] == 1
    prob = P.config5(n=2200, k=32, p=100)
    assert expected_structure_info(prob["A"], prob["cone_dims"], 2200, 100) == dict(
        enabled=1, singleton_rows=2200, empty_rows=0, rest_rows=528, rest_cols=528, compressed=1, base_has_gtg=1)
    assert expected_structure_info(prob["A"], prob["cone_dims"], 2200, 100, aug_rho=0.0)["base_has_gtg"] == 0
    # -0.0 is zero; the threshold is inclusive
    A = np.array([[-0.0, 2.0], [0.0, -0.0], [1.0, 1.0]])
    assert expected_structure_info(A, [("R", 3)], 2, 0) == dict(
        enabled=1, singleton_rows=1, empty_rows=1, rest_rows=1, rest_cols=2, compressed=0, base_has_gtg=0)
    for nJ, compressed in ((512, 1), (513, 0)):
        prob = threshold_problem(nJ)
        assert expected_structure_info(prob["A"], prob["cone_dims"], 1000, 2)["compressed"] == compressed


# ================================================================ 2. GPU cases
@pytest.mark.gpu
def test_scattered_compressed_J():
    prob = scattered_problem()
    info = full_case(prob, 100)
    assert info["compressed"] == 1 and info["rest_cols"] == 150


@pytest.mark.gpu
@pytest.mark.parametrize("fold", [1, 2])
def test_compressed_folded_rest_out_of_global_order(fold):
    prob = folded_problem()
    info = full_case(prob, 200, fold_scaling=fold)
    assert info["compressed"] == 1 and info["rest_cols"] == 150 and info["empty_rows"] > 0


@pytest.mark.gpu
def test_cone_remap_around_dropped_r_cones():
    prob = remap_problem()
    info = full_case(prob, 300)
    assert info["singleton_rows"] == 40 + 10 and info["empty_rows"] == 8 + 10


@pytest.mark.gpu
@pytest.mark.parametrize("nJ,compressed", [(512, 1), (513, 0)])
def test_compression_threshold(nJ, compressed):
    prob = threshold_problem(nJ)
    e = engine(prob)
    info = check_info(e, prob)
    assert info["compressed"] == compressed and info["rest_cols"] == (nJ if compressed else 1000)
    check_H_two_points(e, prob, 400 + nJ)
    check_matvecs(e, prob["A"], 401)
    e.close()


@pytest.mark.gpu
def test_rest_without_columns():
    """Q and S rows of A that are all zero: the rest has rows and J is empty; H = Q + singletons + rho G'G."""
    prob = empty_J_problem()
    e = engine(prob)
    info = check_info(e, prob)
    assert info["rest_rows"] == 7 and info["rest_cols"] == 0 and info["compressed"] == 1
    Fo, ref = check_H_two_points(e, prob, 500)
    n = len(prob["c"])
    x, _ = check_matvecs(e, prob["A"], 501)
    assert np.all(e.mul_A(x)[n:] == 0)
    check_solve(e, prob, Fo, ref, np.random.default_rng(502))
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["q_diag", "q_none", "reg_delta", "aug_rho_0", "torch_A"])
def test_options_on_structured_handle(variant):
    import torch
    prob = scattered_problem(seed=26, n=600, p=4)
    n = len(prob["c"])
    Q, kw, aug_rho, delta, A = "prob", {}, -1.0, 0.0, None
    if variant == "q_diag":
        Q = sp.diags(np.random.default_rng(1).uniform(1.0, 2.0, n)).tocsr()
    elif variant == "q_none":
        Q = None
    elif variant == "reg_delta":
        kw, delta = dict(reg_delta=0.25), 0.25
    elif variant == "aug_rho_0":
        kw, aug_rho = dict(aug_rho=0.0), 0.0
    else:
        A = torch.as_tensor(np.ascontiguousarray(prob["A"].T)).cuda().t()
    e = engine(prob, A=A, Q=Q, **kw)
    info = check_info(e, prob, aug_rho)
    assert info["compressed"] == 1 and info["base_has_gtg"] == (variant != "aug_rho_0")
    Fo, ref = check_H_two_points(e, prob, 600, Q=Q, aug_rho=aug_rho, delta=delta)
    check_matvecs(e, prob["A"], 601)
    if variant == "aug_rho_0":
        check_solve(e, prob, Fo, ref, np.random.default_rng(602), Q=Q)
    e.close()


@pytest.mark.gpu
def test_host_scaling_on_structured_handle():
    """cip_factor with a Diagonal block on every cone, then cip_set_scaling with SymWoodbury blocks on the Q cones
    whose inverse's D differs from the D slot of the cone in front of each (a dropped R cone, the S cone)."""
    import conicip_b200 as cb
    prob = remap_problem()
    cd, A = prob["cone_dims"], prob["A"]
    e = engine(prob)
    rng = np.random.default_rng(700)
    diags = [rng.uniform(0.5, 2.0, k) for _, k in cd]
    assert e.factor(cb.Block([cb.Diagonal(d) for d in diags])) == 0
    Fo = O.Block([O.Diag(d) for d in diags])
    ref = ref_H(prob["Q"], A, prob["G"], cd, Fo, 1.0)
    L = np.tril(e.get_H())                                  # cip_factor leaves the Cholesky factor of H
    assert rel(L @ L.T, ref.H) < 1e-13
    e.form_H()                                              # and the scaling resident
    assert_H(e.get_H(), ref, "factor(Block)")
    check_solve(e, prob, Fo, ref, rng)
    blocks, oblocks = [], []
    for (t, k), d, D in zip(cd, diags, [0.0, 0.5, 0.0, 0.0, 0.0, 2.0]):
        if t == "Q":
            b = 0.3 * rng.standard_normal(k)
            blocks.append(cb.SymWoodbury(d, b, D))
            oblocks.append(O.SymWoodbury(d, b, D))
        else:
            blocks.append(cb.Diagonal(d))
            oblocks.append(O.Diag(d))
    Fo = O.Block(oblocks)
    Zs = [Fo[i].inv().D for i in (1, 5)]
    assert min(abs(z) for z in Zs) > 0.1 and abs(Zs[0] - Zs[1]) > 0.1
    e.set_scaling(cb.Block(blocks))
    e.form_H()
    ref = ref_H(prob["Q"], A, prob["G"], cd, Fo, 1.0)
    assert_H(e.get_H(), ref, "set_scaling")
    check_solve(e, prob, Fo, ref, rng)
    e.close()


# ---------------------------------------------------------------- 8. Julia-style CSC through the C ABI
class RawHandle:
    """The few entry points these tests need, on a handle made by cip_create_csc directly."""

    def __init__(self, h, n, m, p):
        self.h, self.n, self.m, self.p = h, n, m, p

    def _call(self, name, *args):
        from conicip_b200._lib import check, lib
        check(getattr(lib(), name)(self.h, *args))

    def structure_info(self):
        from conicip_b200._lib import StructureInfo
        si = StructureInfo()
        si.struct_size = C.sizeof(StructureInfo)
        self._call("cip_structure_info", C.byref(si))
        return {k: getattr(si, k) for k, _ in StructureInfo._fields_ if k != "struct_size"}

    def nt_scaling(self, v, s):
        lam = np.zeros(self.m)
        self._call("cip_nt_scaling", v.ctypes.data, s.ctypes.data, lam.ctypes.data)

    def form_H(self):
        self._call("cip_form_H")

    def factor_H(self):
        self._call("cip_factor_H")

    def get_H(self):
        out = np.zeros((self.n, self.n), order="F")
        self._call("cip_get_H", out.ctypes.data, self.n)
        return out

    def mul_A(self, x, trans=False):
        y = np.zeros(self.n if trans else self.m)
        self._call("cip_mul_A", int(trans), x.ctypes.data, y.ctypes.data)
        return y

    def solve(self, ry, rw, rv):
        dy, dw, dv = np.zeros(self.n), np.zeros(self.p), np.zeros(self.m)
        self._call("cip_solve", ry.ctypes.data, rw.ctypes.data if self.p else None, rv.ctypes.data, dy.ctypes.data,
                   dw.ctypes.data if self.p else None, dv.ctypes.data)
        return dy, dw, dv

    def close(self):
        from conicip_b200._lib import lib
        lib().cip_destroy(self.h)


def julia_style_csc(A):
    """1-based Int64 CSC of A with row indices in descending order within each column, plus: a duplicate pair
    that sums to an entry of A (two halves), a pair that cancels to exactly 0 in a singleton row (which stays a singleton),
    and a stored -0.0 in an empty row.  Returns (colptr, rowval, nzval)."""
    m, n = A.shape
    cnt = np.count_nonzero(A, axis=1)
    cols = [[(i, A[i, j]) for i in np.flatnonzero(A[:, j])] for j in range(n)]
    i2 = int(np.flatnonzero(cnt >= 2)[0])
    j2 = int(np.flatnonzero(A[i2])[0])
    cols[j2] = [(i, x / 2 if i == i2 else x) for i, x in cols[j2]] + [(i2, A[i2, j2] / 2)]
    i1 = int(np.flatnonzero(cnt == 1)[0])
    j1 = int(np.flatnonzero(A[i1] == 0)[0])
    cols[j1] += [(i1, 0.7), (i1, -0.7)]
    i0 = int(np.flatnonzero(cnt == 0)[0])
    cols[0] += [(i0, -0.0)]
    cp, rv, nz = [1], [], []
    for c in cols:
        c = sorted(c, key=lambda e: -e[0])            # stable: duplicates stay in the order above
        rv += [i + 1 for i, _ in c]
        nz += [x for _, x in c]
        cp.append(cp[-1] + len(c))
    return np.array(cp, np.int64), np.array(rv, np.int64), np.array(nz, np.float64)


@pytest.mark.gpu
def test_julia_style_csc_matches_dense_input_bitwise():
    import conicip_b200 as cb
    from conicip_b200._lib import Csc, Options, lib
    prob = remap_problem()
    Q, A, G, cd = prob["Q"], prob["A"], prob["G"], prob["cone_dims"]
    m, n, p = A.shape[0], A.shape[1], G.shape[0]
    keep = []

    def csc(arrays, shape):
        keep.extend(arrays)
        cp, rv, nz = arrays
        return Csc(shape[0], shape[1], cp.ctypes.data, rv.ctypes.data, nz.ctypes.data, 1)

    def julia(M):
        M = sp.csc_matrix(M)
        return csc(((M.indptr + 1).astype(np.int64), (M.indices + 1).astype(np.int64), M.data.astype(np.float64)),
                   M.shape)

    arrays = julia_style_csc(A)
    # the arrays hold exactly A once duplicates are summed in storage order
    S = sp.csc_matrix((arrays[2], arrays[1] - 1, arrays[0] - 1), shape=A.shape)
    assert np.array_equal(S.toarray(), A)
    ct = np.array([cb.CONE_R if t == "R" else cb.CONE_Q if t == "Q" else cb.CONE_S for t, _ in cd], dtype=np.int32)
    cdim = np.array([k for _, k in cd], dtype=np.int32)
    o = Options()
    o.struct_size = C.sizeof(Options)
    o.device, o.aug_rho, o.dist_chol, o.row_structure = -1, -1.0, -1, 1
    h = C.c_void_p()
    qs, as_, gs = julia(Q), csc(arrays, A.shape), julia(G)
    rc = lib().cip_create_csc(C.byref(h), n, C.byref(qs), C.byref(as_), C.byref(gs), len(cd), ct.ctypes.data,
                              cdim.ctypes.data, C.byref(o))
    assert rc == 0, cb._lib.last_error()
    e_csc = RawHandle(h, n, m, p)
    e_dense = engine(prob)
    assert e_csc.structure_info() == e_dense.structure_info() == expected_structure_info(A, cd, n, p)
    rng = np.random.default_rng(801)
    x, u = rng.standard_normal(n), rng.standard_normal(m)
    for e in (e_csc, e_dense):
        assert_matvec(e.mul_A(x), A, x)
    assert np.array_equal(e_csc.mul_A(x), e_dense.mul_A(x))
    assert np.array_equal(e_csc.mul_A(u, trans=True), e_dense.mul_A(u, trans=True))
    v, s = cone_point(cd, rng), cone_point(cd, rng)
    Hs = []
    for e in (e_csc, e_dense):
        e.nt_scaling(v, s)
        e.form_H()
        Hs.append(e.get_H())
    assert np.array_equal(Hs[0], Hs[1])
    assert_H(Hs[0], ref_H(Q, A, G, cd, oracle_F(cd, v, s), 1.0), "CSC")
    ry, rw, rv = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(m)
    outs = []
    for e in (e_csc, e_dense):
        e.factor_H()
        outs.append(e.solve(ry, rw, rv))
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    Fo = oracle_F(cd, v, s)
    oy, ow, ov = O.kktsolver_qr(Q, A, G, cd)(Fo, Fo.inv_adjoint())(ry, rw, rv)
    assert rel(outs[0][0], oy) < 1e-9 and rel(outs[0][2], ov) < 1e-9 and rel(outs[0][1], ow) < 1e-8
    e_csc.close()
    e_dense.close()


# ---------------------------------------------------------------- 9. sizes
def ragged_problem(n, m, seed):
    """A Q cone of dense rows, then an R cone whose last rows (in the ragged last quad of rows) are empty,
    two-non-zero and singleton rows."""
    rng = np.random.default_rng(seed)
    rows = list(rng.standard_normal((3, n)) / np.sqrt(n))
    kinds = [0, 1, 2] if n > 1 else [0, 1]                  # n = 1: empty and singleton rows only
    for t in range(m - 3):
        kd = kinds[t % len(kinds)]
        rows.append(np.zeros(n) if kd == 0 else sparse_row(n, rng.choice(n, 1 if kd == 1 else 2, replace=False), rng))
    return finish("ragged", np.array(rows), [("Q", 3), ("R", m - 3)], 0, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 129, 131])
def test_ragged_row_counts(n):
    for r in (1, 2, 3):
        m = 200 + r
        prob = ragged_problem(n, m, seed=900 + n + r)
        assert m % 4 == r
        e = engine(prob)
        check_info(e, prob)
        check_H_two_points(e, prob, 901 + r)
        check_matvecs(e, prob["A"], 902)
        e.close()


@pytest.mark.gpu
def test_rest_of_more_than_65535_rows():
    rng = np.random.default_rng(950)
    n, nr = 64, 70000
    A = np.zeros((nr + n, n))
    A[np.arange(n), np.arange(n)] = rng.uniform(0.5, 2.0, n)
    c0 = rng.integers(0, n, nr)
    c1 = (c0 + rng.integers(1, n, nr)) % n
    A[n + np.arange(nr), c0] = rng.standard_normal(nr)
    A[n + np.arange(nr), c1] = rng.standard_normal(nr)
    prob = finish("tall_rest", A, [("R", nr + n)], 0, rng)
    e = engine(prob)
    info = check_info(e, prob)
    assert info["rest_rows"] == nr and info["singleton_rows"] == n
    check_H_two_points(e, prob, 951)
    rng = np.random.default_rng(952)
    x = rng.standard_normal(n)
    assert_matvec(e.mul_A(x), A, x, "A x")
    e.close()


# ---------------------------------------------------------------- 10. whole solves against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["folded", "remap"])
def test_full_solve_against_oracle(name):
    import conicip_b200 as cb
    prob = folded_problem() if name == "folded" else remap_problem()
    Q, c, A, b, cd, G, d = (prob[k] for k in ("Q", "c", "A", "b", "cone_dims", "G", "d"))
    so = O.conicIP(Q, c, A, b, cd, G, d, optTol=1e-8, kktsolver=oracle_kkt(prob))
    eng = engine(prob, fold_scaling=1) if name == "folded" else None
    s = cb.conicIP_native(Q, c, A, b, cd, G, d, engine=eng, row_structure=1, optTol=1e-8)
    if eng is not None:
        assert eng.structure_info()["compressed"] == 1
        eng.close()
    assert s.status == so.status == "Optimal" and abs(s.Iter - so.Iter) <= 1, (s.status, s.Iter, so.Iter)
    for f in ("y", "v", "w"):
        assert rel(getattr(s, f), getattr(so, f)) < 1e-6, f
    assert max(s.prFeas, s.duFeas, s.muFeas) < 1e-8
