"""cip_options.eliminate_y: the m-space form of the KKT system (factor M = F'F + A D^-1 A', D = Q + delta I).

M is checked elementwise against an FP64 reference built from the oracle's own scaling blocks (R, Woodbury and S,
with an S cone of order 8); the KKT solves against the oracle's kktsolver_qr and the 3x3 residual; whole solves
against the oracle's conicIP and against the n-space form on the same problem; the rejections; and the reach case
for which the option exists: a wide problem whose n x n H would need 180 GB.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import oracle as O
from test_gpu_row_structure_reference import cone_point, oracle_F

U = 2.0 ** -53

# C_M: |M_dev - M_ref| <= C_M * u * (n + 2) * B elementwise, B = B_F + |A| D^-1 |A|'.  The constant part A D^-1 A' is a
# sum of n products (gamma_n = n u / (1 - n u) times |A| D^-1 |A|', Higham, Accuracy and Stability, sec. 3.1), made
# once by the device and once by the reference.  F'F is made by the device from the closed forms of
# csrc/eliminate_y.cu (a few operations per entry, and for S cones W = R R', a sum of k products) and by the
# reference as F_dense' F_dense; both are within a few u of B_F, the same closed form with every term replaced by its
# absolute value (|R||R|' for W) -- the bound of the computed expression, which |F|'|F| is not where the Woodbury
# terms cancel.  The two scalings are computed independently from the same (v, s) and differ by a few ulps per entry.
# That is at most 2 * 2 gamma_n plus a few u in all: C_M = 4 with the "+ 2".  A wrong entry (a sign, a missing
# sqrt(2), D^-1 applied twice) is wrong by a sizeable fraction of B.
C_M = 4

CONES = [("R", 40), ("Q", 9), ("R", 3), ("S", 36), ("Q", 33), ("R", 17), ("S", 6)]      # S of order 8 and 3; m = 144


@pytest.fixture(autouse=True)
def _option_decides(monkeypatch):
    for k in ("CIP_ROW_STRUCTURE", "CIP_FOLD_SCALING", "CIP_FAST_SYRK"):
        monkeypatch.delenv(k, raising=False)


def cbm():
    import conicip_b200 as cb
    return cb


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def host(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def m_of(cones):
    return sum(k for _, k in cones)


# ================================================================ reference
def svec_pairs(k):
    """(i, j), i <= j, in the order of the engine's svec (row-major upper triangle, csrc/sdp.cu)."""
    return [(i, j) for i in range(k) for j in range(i, k)]


def block_bound(b):
    """Term-wise absolute bound of the device's closed form of F_b' F_b."""
    if isinstance(b, O.Diag):
        return np.diag(b.diag ** 2)
    if isinstance(b, O.SymWoodbury):
        a, v, D = b.Adiag, b.B, b.D
        ab = np.abs(a * v)
        return (np.diag(a ** 2) + abs(D) * (np.outer(ab, np.abs(v)) + np.outer(np.abs(v), ab))
                + D * D * float(v @ v) * np.outer(np.abs(v), np.abs(v)))
    k = b.R.shape[0]
    V = np.abs(b.R) @ np.abs(b.R).T
    pr = svec_pairs(k)
    kap = np.array([np.sqrt(0.5) if i == j else 1.0 for i, j in pr])
    I = np.array([i for i, _ in pr])
    J = np.array([j for _, j in pr])
    return np.outer(kap, kap) * (V[I][:, I] * V[J][:, J] + V[I][:, J] * V[J][:, I])


def ref_M(A, d, F):
    """M = F'F + A D^-1 A' in float64 from the oracle's blocks, and its bound matrix B."""
    A = A.toarray() if sp.issparse(A) else np.asarray(A)
    Fd = F.dense()
    m = A.shape[0]
    BF = np.zeros((m, m))
    for i, b in enumerate(F.blocks):
        lo, hi = F.offsets[i], F.offsets[i + 1]
        BF[lo:hi, lo:hi] = block_bound(b)
    M = Fd.T @ Fd + (A / d) @ A.T
    B = BF + (np.abs(A) / d) @ np.abs(A).T
    return M, B


def assert_M(M, ref, A, what):
    Mr, B = ref
    tol = C_M * U * (A.shape[1] + 2) * B
    bad = np.tril(~(np.abs(M - Mr) <= tol))
    if bad.any():
        i, j = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {int(bad.sum())} entries of M outside the bound, first M[{i},{j}] = "
                             f"{M[i, j]!r}, reference {Mr[i, j]!r}, bound {tol[i, j]:.3e}")


def cb_block(F):
    cb = cbm()
    out = []
    for b in F.blocks:
        if isinstance(b, O.Diag):
            out.append(cb.Diagonal(b.diag))
        elif isinstance(b, O.SymWoodbury):
            out.append(cb.SymWoodbury(b.Adiag, b.B, b.D))
        else:
            out.append(cb.VecCongurance(b.R))
    return cb.Block(out)


# ================================================================ problems
def make(cones=CONES, n=600, p=0, seed=0):
    rng = np.random.default_rng(seed)
    m = m_of(cones)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    G = rng.standard_normal((p, n)) / np.sqrt(n) if p else None
    q = rng.uniform(0.5, 2.0, n)
    return A, G, q


def engine(A, G, q, qkind, akind, cones=CONES, delta=0.0, **kw):
    """qkind: 'diag' (q_kind 1), 'dense' (a dense diagonal Q), 'zero' (Q = 0); akind: 'dense', 'csc', 'torch'."""
    cb = cbm()
    n = A.shape[1]
    if akind == "csc":
        Q = None if qkind == "zero" else sp.diags(q).tocsc()
        Aa, Ga = sp.csc_matrix(A), (None if G is None else sp.csc_matrix(G))
    else:
        Q = {"diag": sp.diags(q), "dense": np.diag(q), "zero": None}[qkind]
        Ga = G
        Aa = A
        if akind == "torch":
            import torch
            Aa = torch.tensor(np.ascontiguousarray(A.T), device="cuda").t()
    e = cb.Engine(Q, Aa, Ga, cones, reg_delta=delta, **kw)
    assert e.n == n
    return e


def d_of(q, qkind, delta):
    return (np.zeros_like(q) if qkind == "zero" else q) + delta


# ================================================================ 1. M against the FP64 reference
@pytest.mark.gpu
@pytest.mark.parametrize("p", [0, 6])
def test_M_against_fp64_reference(p):
    cb = cbm()
    A, G, q = make(p=p, seed=1)
    e = engine(A, G, q, "diag", "dense", delta=0.0, eliminate_y=1)
    assert e.kkt_form_info() == {"eliminate_y": 1, "automatic": 0}
    rng = np.random.default_rng(2)
    d = q.copy()
    for wide in (False, True):
        v, s = cone_point(CONES, rng, wide), cone_point(CONES, rng, wide)
        if wide:      # the NT scaling of the wide point spans v / s from 1e-8 to 1e8
            vs = v[:40] / s[:40]
            assert vs.min() < 1e-3 and vs.max() > 1e3
        F = oracle_F(CONES, v, s)
        e.nt_scaling(v, s)
        e.form_H()
        assert_M(e.get_M(), ref_M(A, d, F), A, f"NT scaling {'wide' if wide else 'central'}")
        # the same F supplied by the host as a Block
        e.set_scaling(cb_block(F))
        e.form_H()
        assert_M(e.get_M(), ref_M(A, d, F), A, "host Block")
    # F = I, the first call of conicIP (DIAG blocks of ones in every slot, Q and S included)
    ones = O.Block([O.Diag(np.ones(k)) for _, k in CONES])
    e.set_scaling(cb.Block([cb.Diagonal(np.ones(k)) for _, k in CONES]))
    e.form_H()
    assert_M(e.get_M(), ref_M(A, d, ones), A, "F = I")
    st = e.stats()
    assert st["syrk_flops"] == 0.0
    # after the factorisation get_M shows L with L L' = M
    v, s = cone_point(CONES, rng), cone_point(CONES, rng)
    Mr, _ = ref_M(A, d, oracle_F(CONES, v, s))
    e.factor_from_point(v, s)
    L = np.tril(e.get_M())
    assert rel(L @ L.T, Mr) < 1e-12
    st = e.stats()
    m = A.shape[0]
    assert st["chol_flops"] == pytest.approx(m ** 3 / 3.0)
    assert st["syrk_flops"] == 0.0


# ================================================================ 2. KKT solves
SOLVE_CASES = [("diag", "dense", 0.0), ("dense", "dense", 0.25), ("zero", "dense", 0.5), ("diag", "csc", 0.0),
               ("diag", "torch", 1e-3), ("zero", "csc", 0.75)]


@pytest.mark.gpu
@pytest.mark.parametrize("qkind,akind,delta", SOLVE_CASES)
@pytest.mark.parametrize("p", [0, 7])
def test_kkt_solves(qkind, akind, delta, p):
    A, G, q = make(p=p, seed=3 + p)
    n, m = A.shape[1], A.shape[0]
    Gd = G if p else np.zeros((0, n))
    e = engine(A, G, q, qkind, akind, delta=delta, eliminate_y=1)
    assert e.kkt_form_info()["eliminate_y"] == 1
    d = d_of(q, qkind, delta)
    Qref = np.diag(d)
    rng = np.random.default_rng(5)
    v, s = cone_point(CONES, rng), cone_point(CONES, rng)
    F = oracle_F(CONES, v, s)
    assert e.factor_from_point(v, s) is not None and e.last_factor_status == 0
    ry, rw, rv = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(m)
    dy, dw, dv = e.solve(ry, rw if p else None, rv)
    # against the oracle's double-QR kktsolver
    x, y, z = O.kktsolver_qr(Qref, A, Gd, CONES)(F, F.inv_adjoint())(ry, rw, rv)
    assert rel(dy, x) < 1e-9 and rel(dv, z) < 1e-9
    if p:
        assert rel(dw, y) < 1e-9
    # the 3x3 residual:  Q a + G'b - A'c = ry ;  G a = rw ;  A a + F'F c = rv   (D = Q + delta I)
    Fd = F.dense()
    W = Fd.T @ Fd
    r1 = Qref @ dy + Gd.T @ dw - A.T @ dv - ry
    r3 = A @ dy + W @ dv - rv
    scale = np.linalg.norm(ry) + np.linalg.norm(rv) + np.linalg.norm(Qref @ dy) + np.linalg.norm(W @ dv)
    assert np.linalg.norm(r1) < 1e-11 * scale and np.linalg.norm(r3) < 1e-11 * scale
    if p:
        assert np.linalg.norm(Gd @ dy - rw) < 1e-11 * (np.linalg.norm(rw) + np.linalg.norm(dy))
    # solve_multi equals solve column by column, bit for bit (also with an odd column count)
    RY, RW, RV = (np.asfortranarray(rng.standard_normal(sh)) for sh in ((n, 3), (p, 3), (m, 3)))
    MY, MW, MV = e.solve_multi(RY, RW if p else None, RV)
    for k in range(3):
        sy, sw, sv = e.solve(RY[:, k], RW[:, k] if p else None, RV[:, k])
        assert np.array_equal(MY[:, k], sy) and np.array_equal(MV[:, k], sv)
        if p:
            assert np.array_equal(MW[:, k], sw)
    # deterministic: the same solve again, and again after a fresh factorisation at the same point
    assert all(np.array_equal(a, b) for a, b in zip(e.solve(ry, rw if p else None, rv), (dy, dw, dv)))
    e.factor_from_point(v, s)
    assert all(np.array_equal(a, b) for a, b in zip(e.solve(ry, rw if p else None, rv), (dy, dw, dv)))
    # solve_H keeps its meaning: H^-1 rhs with H = D + A'(F'F)^-1 A
    H = Qref + A.T @ np.linalg.solve(W, A)
    rhs = rng.standard_normal(n)
    assert rel(e.solve_H(rhs), np.linalg.solve(H, rhs)) < 1e-9
    # the resident operators: A and G as given, Q without delta
    xn, xm = rng.standard_normal(n), rng.standard_normal(m)
    assert rel(e.mul_A(xn), A @ xn) < 1e-13 and rel(e.mul_A(xm, trans=True), A.T @ xm) < 1e-13
    Qy = e.mul_Q(xn)
    assert rel(Qy, (d - delta) * xn) < 1e-15 if qkind != "zero" else np.all(Qy == 0.0)
    if p:
        xp = rng.standard_normal(p)
        assert rel(e.mul_G(xn), G @ xn) < 1e-13 and rel(e.mul_G(xp, trans=True), G.T @ xp) < 1e-13


@pytest.mark.gpu
def test_device_vectors_and_n_space_agree():
    """torch vectors in and out, and the same solve through the n-space form (eliminate_y = 2)"""
    import torch
    A, G, q = make(p=5, seed=9)
    n, m = A.shape[1], A.shape[0]
    ey = engine(A, G, q, "diag", "torch", eliminate_y=1)
    en = engine(A, G, q, "diag", "dense", eliminate_y=2)
    assert en.kkt_form_info() == {"eliminate_y": 0, "automatic": 0}
    rng = np.random.default_rng(4)
    v, s = cone_point(CONES, rng), cone_point(CONES, rng)
    for e in (ey, en):
        e.factor_from_point(v, s)
    ry, rw, rv = rng.standard_normal(n), rng.standard_normal(5), rng.standard_normal(m)
    T = lambda x: torch.tensor(x, device="cuda")
    got = ey.solve(T(ry), T(rw), T(rv))
    assert all(isinstance(g, torch.Tensor) and g.is_cuda for g in got)
    for a, b in zip(got, en.solve(ry, rw, rv)):
        assert rel(host(a), b) < 1e-9


# ================================================================ 3. full solves
def wide_problem(seed=11, n=900, p=5):
    rng = np.random.default_rng(seed)
    cones = [("R", 60), ("Q", 17), ("S", 36), ("R", 20), ("Q", 33), ("S", 10)]
    m = m_of(cones)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    y0 = rng.standard_normal(n)
    b = A @ y0 - cone_point(cones, rng)
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    q = rng.uniform(0.5, 2.0, n)
    return dict(Q=sp.diags(q).tocsr(), c=rng.standard_normal(n), A=A, b=b, cone_dims=cones, G=G, d=G @ y0)


@pytest.mark.gpu
def test_full_solves_against_oracle_and_n_space():
    cb = cbm()
    pr = wide_problem()
    args = (pr["Q"], pr["c"], pr["A"], pr["b"], pr["cone_dims"], pr["G"], pr["d"])
    so = O.conicIP(pr["Q"].toarray(), *args[1:], optTol=1e-8)
    assert so.status == "Optimal"
    runs = {"native m-space": cb.conicIP_native(*args, eliminate_y=1, optTol=1e-8),
            "host m-space": cb.conicIP(*args, eliminate_y=1, optTol=1e-8),
            "native n-space": cb.conicIP_native(*args, eliminate_y=2, optTol=1e-8)}
    for name, s in runs.items():
        assert s.status == so.status, (name, s.status)
        assert abs(s.Iter - so.Iter) <= 1, (name, s.Iter, so.Iter)
        for f in ("y", "w", "v"):
            a, b = host(getattr(s, f)), getattr(so, f)
            assert np.max(np.abs(a - b)) <= 1e-6 * max(1.0, np.max(np.abs(b))), (name, f)
    a, b = runs["native m-space"], runs["native n-space"]
    assert abs(a.Iter - b.Iter) <= 1
    assert rel(a.y, b.y) < 1e-6 and rel(a.v, b.v) < 1e-6


# ================================================================ 4. loud rejections, pivot failures
@pytest.mark.gpu
def test_rejections():
    cb = cbm()
    A, G, q = make(p=3, seed=6)
    n = A.shape[1]
    Qoff = np.diag(q)
    Qoff[3, 17] = Qoff[17, 3] = 0.1
    with pytest.raises(cb.CipError, match="off-diagonal"):
        cb.Engine(Qoff, A, G, CONES, eliminate_y=1)
    with pytest.raises(cb.CipError, match="off-diagonal"):
        cb.Engine(sp.csc_matrix(Qoff), sp.csc_matrix(A), sp.csc_matrix(G), CONES, eliminate_y=1)
    qneg = q.copy()
    qneg[5] = -1.0
    with pytest.raises(cb.CipError, match="reg_delta"):
        cb.Engine(sp.diags(qneg), A, G, CONES, eliminate_y=1, reg_delta=0.5)
    with pytest.raises(cb.CipError, match="reg_delta"):
        cb.Engine(None, A, G, CONES, eliminate_y=1)                   # Q = 0 needs reg_delta > 0
    with pytest.raises(cb.CipError, match="row_structure"):
        cb.Engine(sp.diags(q), A, G, CONES, eliminate_y=1, row_structure=1)
    with pytest.raises(cb.CipError, match="single-device"):
        cb.Engine(sp.diags(q), A, G, CONES, eliminate_y=1, ngpus=2)
    # the same Q with the default: an ordinary n-space handle (it fits)
    e = cb.Engine(Qoff, A, G, CONES)
    assert e.kkt_form_info() == {"eliminate_y": 0, "automatic": 0}
    with pytest.raises(cb.CipError, match="cip_get_H"):
        e.get_M()
    ey = cb.Engine(sp.diags(q), A, G, CONES, eliminate_y=1)
    with pytest.raises(cb.CipError, match="cip_get_M"):
        ey.get_H()
    with pytest.raises(cb.CipError, match="single-device"):
        ey.comm_init(2, 0, bytes(128))
    assert n > 0


@pytest.mark.gpu
def test_pivot_failures_report_documented_index():
    cb = cbm()
    A, G, q = make(p=6, seed=7)
    m = A.shape[0]
    # M: a zero row of A with a zero scaling there leaves M_rr = 0 -> 1 + row of A
    A0 = A.copy()
    A0[57] = 0.0
    e = cb.Engine(sp.diags(q), A0, G, CONES, eliminate_y=1)
    a = np.ones(m)
    a[57] = 0.0
    blocks, off = [], 0
    for _, k in CONES:
        blocks.append(cb.Diagonal(a[off:off + k]))
        off += k
    assert e.factor(cb.Block(blocks)) == 58
    # S: a zero row of G leaves S_rr = P_rr - (Z Z')_rr = 0 -> m + 1 + row of G
    G0 = G.copy()
    G0[3] = 0.0
    e = cb.Engine(sp.diags(q), A, G0, CONES, eliminate_y=1)
    assert e.factor(cb.Block([cb.Diagonal(np.ones(k)) for _, k in CONES])) == m + 4


# ================================================================ 5. reach
@pytest.mark.gpu
def test_reach_wide_problem_auto():
    """n = 150 000, m = 2 048 dense, Q = I, p = 64: the n x n H alone would take n_pad^2 * 8 = 180 GB (twice, with
    Q), so the default option must choose the m-space form, and the problem must solve."""
    import torch
    cb = cbm()
    n, p = 150_000, 64
    cones = [("R", 1024)] + [("Q", 64)] * 16
    m = m_of(cones)
    n_pad = (n + 127) // 128 * 128
    assert 2 * n_pad * n_pad * 8 > 2 * 170e9          # the n-space form: Qq4 and H4 (shapes only, never run)
    g = torch.Generator(device="cuda").manual_seed(20261022)
    At = torch.randn((n, m), generator=g, device="cuda", dtype=torch.float64) / np.sqrt(n)    # A = At.t(), col-major
    Gt = torch.randn((n, p), generator=g, device="cuda", dtype=torch.float64) / np.sqrt(n)
    A, G = At.t(), Gt.t()
    y0 = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    s0 = torch.tensor(cone_point(cones, np.random.default_rng(1)), device="cuda")
    b = A @ y0 - s0
    d = G @ y0
    c = torch.randn(n, generator=g, device="cuda", dtype=torch.float64)
    e = cb.Engine(sp.identity(n, format="csr"), A, G, cones)
    assert e.kkt_form_info() == {"eliminate_y": 1, "automatic": 1}
    st = e.stats()
    # A once (m_pad x n_pad) plus G, the split-K workspace, M and C, vectors: far below one n x n buffer
    assert st["device_bytes"] < 1.3 * m * n_pad * 8 + 1.0e9, st["device_bytes"]
    y, w, v, info = e.ipm_solve(c, b, d, optTol=1e-8)
    assert info["status"] == "Optimal", info
    # residuals recomputed on the device (Q = I)
    nc, nb, nd = float(c.norm()), float(b.norm()), float(d.norm())
    rdu = float((y + G.t() @ w - A.t() @ v - c).norm()) / (1 + nc)
    req = float((G @ y - d).norm()) / (1 + nd)
    sl = A @ y - b
    rr = float(torch.clamp(-sl[:1024], min=0).max()) / (1 + nb)
    qs = sl[1024:].reshape(16, 64)
    rq = float(torch.clamp(qs[:, 1:].norm(dim=1) - qs[:, 0], min=0).max()) / (1 + nb)
    gap = abs(float(v @ sl)) / (1 + abs(float(c @ y)))
    assert max(rdu, req, rr, rq) < 1e-7, (rdu, req, rr, rq)
    assert gap < 1e-6, gap
    e.close()


# ================================================================ 6. default unchanged
@pytest.mark.gpu
def test_default_handle_keeps_the_n_space_form():
    cb = cbm()
    A, G, q = make(p=2, seed=8)
    for Q in (sp.diags(q), np.diag(q), sp.diags(q).tocsc()):
        e = cb.Engine(Q, A, G, CONES)
        assert e.kkt_form_info() == {"eliminate_y": 0, "automatic": 0}
        e.get_H()
