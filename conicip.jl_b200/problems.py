"""Synthetic problem generators: the reference's deterministic test problems and the
BASELINE.json configurations C1..C4 (SURVEY.md section 8d).

Julia's RNG stream is not reproducible here, so "identical inputs" for the oracle and the
engine means: both consume the arrays produced by these NumPy (PCG64) generators.
Every problem is a dict: Q, c, A, b, cone_dims, G, d (+ name and notes).
"""
import numpy as np
import scipy.sparse as sp


def _prob(name, Q, c, A, b, cone_dims, G=None, d=None, **kw):
    n = len(c)
    if G is None:
        G = np.zeros((0, n))
        d = np.zeros(0)
    out = dict(name=name, Q=Q, c=np.asarray(c, float), A=A, b=np.asarray(b, float),
               cone_dims=list(cone_dims), G=G, d=np.asarray(d, float))
    out.update(kw)
    return out


# ------------------------------------------------------------------ reference test problems
def sphere(n=2):
    """test/runtests.jl:137-166 -- projection onto the unit ball (one Q cone)."""
    H = np.eye(n)
    a = np.ones(n)
    A = np.vstack([np.zeros((1, n)), np.eye(n)])
    b = np.concatenate([[-1.0], np.zeros(n)])
    return _prob("sphere", H, H @ a, A, b, [("Q", n + 1)], optTol=1e-7)


def combined(n=10):
    """test/runtests.jl:168-206 -- R^n x Q^(n+1)."""
    H = np.eye(n)
    c = np.arange(1.0, n + 1)
    A = np.vstack([np.eye(n), np.zeros((1, n)), np.eye(n)])
    b = np.concatenate([np.zeros(n), [-1.0], np.zeros(n)])
    return _prob("combined", H, H @ c, A, b, [("R", n), ("Q", n + 1)], optTol=1e-7)


def simplex(n=10):
    """test/runtests.jl:208-244 -- projection onto the simplex (R^n + one equality)."""
    H = np.eye(n)
    c = np.arange(1.0, n + 1)
    return _prob("simplex", H, H @ c, np.eye(n), np.zeros(n), [("R", n)], np.ones((1, n)), [1.0], optTol=1e-7)


def box_qp(n=1000):
    """test/runtests.jl:90-131 -- box-constrained QP, H = 0.5 I."""
    H = 0.5 * np.eye(n)
    c = np.arange(1.0, n + 1)
    A = np.vstack([np.eye(n), -np.eye(n)])
    b = -np.ones(2 * n)
    return _prob("box_qp", H, H @ c, A, b, [("R", 2 * n)], optTol=1e-7)


def soc_direct():
    """test/runtests.jl:554-590 -- Q^4 x R^4."""
    n = 4
    Q = np.eye(n)
    c = -np.ones(n)
    A_soc = np.vstack([np.zeros((1, n)), np.eye(n)[:3]])
    A = np.vstack([A_soc, np.eye(n)])
    b = np.concatenate([[-1.0, 0, 0, 0], np.zeros(n)])
    return _prob("soc_direct", Q, c, A, b, [("Q", 4), ("R", n)], optTol=1e-6)


def moi_simple_lp():
    """`Simple LP via MOI` (test/runtests.jl:684-715) as the wrapper hands it to conicIP (src/MOI_wrapper.jl:142-285):
    min x1 + x2  s.t.  x1 + x2 >= 1, x >= 0; objective 1, x = (0.5, 0.5) (analytic centre of the optimal face)."""
    A = np.array([[1.0, 1.0], [1.0, 0.0], [0.0, 1.0]])
    return _prob("moi_simple_lp", np.zeros((2, 2)), -np.array([1.0, 1.0]), A, np.array([1.0, 0.0, 0.0]), [("R", 3)], optTol=1e-6)


def moi_soc():
    """`SOC via MOI` (test/runtests.jl:717-744): min x3  s.t.  x1 = 1, x2 = 1, ||(x1, x2)|| <= x3; x3 = sqrt(2)."""
    A = np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])
    G = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])
    return _prob("moi_soc", np.zeros((3, 3)), -np.array([0.0, 0.0, 1.0]), A, np.zeros(3), [("Q", 3)], G, np.array([1.0, 1.0]),
                 optTol=1e-6)


def moi_max_sense():
    """`Max sense via MOI` (test/runtests.jl:746-775): max x1 + 2 x2  s.t.  x1 + x2 <= 1, x >= 0; objective 2, x = (0, 1)."""
    A = np.array([[-1.0, -1.0], [1.0, 0.0], [0.0, 1.0]])
    return _prob("moi_max_sense", np.zeros((2, 2)), np.array([1.0, 2.0]), A, np.array([-1.0, 0.0, 0.0]), [("R", 3)], optTol=1e-6)


def infeasible(n=10, seed=0):
    """test/runtests.jl:441-460 (shape only; data from NumPy's RNG)."""
    rng = np.random.default_rng(seed)
    h = rng.standard_normal(n)
    H = np.outer(h, h)
    c = np.arange(1.0, n + 1)
    A = np.vstack([np.eye(n), -np.eye(n)])
    b = np.ones(2 * n)
    return _prob("infeasible", H, H @ c, A, b, [("R", 2 * n)], optTol=1e-7)


def unbounded(n=10):
    """test/runtests.jl:487-505."""
    return _prob("unbounded", np.zeros((n, n)), np.arange(1.0, n + 1), np.eye(n), np.zeros(n), [("R", n)],
                 optTol=1e-7)


# ------------------------------------------------------------------ BASELINE configurations
def _lowrank_q(rng, n, r=32):
    U = rng.standard_normal((n, r)) / np.sqrt(r)
    return np.diag(rng.uniform(1.0, 2.0, n)) + U @ U.T


def config1(n=1000, seed=1):
    """C1 -- README QP: Q = S'S with S ~ sprandn(n,n,0.1), c = 1, A = I, K = R^n (README.md:59-68)."""
    rng = np.random.default_rng(seed)
    S = sp.random(n, n, density=0.1, random_state=rng, data_rvs=rng.standard_normal, format="csr")
    Q = (S.T @ S).toarray()
    return _prob("C1", Q, np.ones(n), np.eye(n), np.zeros(n), [("R", n)], optTol=1e-8)


def config2(n=8192, m=16384, seed=2):
    """C2 -- dense polyhedral QP, K = R^m (strictly feasible by construction)."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    y0 = rng.standard_normal(n)
    s0 = rng.uniform(0.1, 1.1, m)
    b = A @ y0 - s0
    Q = _lowrank_q(rng, n)
    c = rng.standard_normal(n)
    return _prob("C2", Q, c, A, b, [("R", m)], optTol=1e-8)


def config3(n=4096, ncones=512, k=33, p=256, seed=3):
    """C3 -- SOCP: `ncones` Q cones of dim k plus an equality block G (p rows)."""
    rng = np.random.default_rng(seed)
    m = ncones * k
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    y0 = rng.standard_normal(n)
    s0 = np.zeros(m)
    for i in range(ncones):
        u = 0.1 * rng.standard_normal(k - 1)
        s0[i * k] = 1.0 + np.linalg.norm(u)
        s0[i * k + 1:(i + 1) * k] = u
    b = A @ y0 - s0
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    d = G @ y0
    Q = _lowrank_q(rng, n)
    c = rng.standard_normal(n)
    return _prob("C3", Q, c, A, b, [("Q", k)] * ncones, G, d, optTol=1e-8)


def mixed(n=96, mr=80, ncones=6, k=9, p=5, seed=7):
    """Small R + Q + equality problem exercising every R/Q code path (tests)."""
    rng = np.random.default_rng(seed)
    m = mr + ncones * k
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    y0 = rng.standard_normal(n)
    s0 = np.zeros(m)
    s0[:mr] = rng.uniform(0.1, 1.1, mr)
    for i in range(ncones):
        o = mr + i * k
        u = 0.1 * rng.standard_normal(k - 1)
        s0[o] = 1.0 + np.linalg.norm(u)
        s0[o + 1:o + k] = u
    b = A @ y0 - s0
    G = rng.standard_normal((p, n)) / np.sqrt(n)
    d = G @ y0
    Q = _lowrank_q(rng, n, 8)
    c = rng.standard_normal(n)
    cones = ([("R", mr)] if mr > 0 else []) + [("Q", k)] * ncones
    return _prob("mixed", Q, c, A, b, cones, G, d, optTol=1e-8)


def config4_device(n=16384, m=262144, seed=4, rank=0, nranks=1, scale_rows=None):
    """C4 -- large dense QP generated directly on the device, row-sharded: this rank's slab
    holds rows [rank*m/nranks, (rank+1)*m/nranks).  Rows are drawn from a per-row-block
    Philox stream so every sharding sees the same global matrix.
    Returns torch tensors: At (n x m_local, contiguous => column-major A slab), b, Q (dense, symmetric; `qdiag` is
    its diagonal part), c."""
    import torch
    m_loc = m // nranks
    r0 = rank * m_loc
    blk = 4096
    At = torch.empty((n, m_loc), dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda")
    for i0 in range(0, m_loc, blk):
        g.manual_seed(seed * 1_000_003 + (r0 + i0) // blk)
        nb = min(blk, m_loc - i0)
        At[:, i0:i0 + nb] = torch.randn((n, nb), generator=g, dtype=torch.float64, device="cuda") / (n ** 0.5)
    g.manual_seed(seed)
    y0 = torch.randn(n, generator=g, dtype=torch.float64, device="cuda")
    c = torch.randn(n, generator=g, dtype=torch.float64, device="cuda")
    qdiag = 1.0 + torch.rand(n, generator=g, dtype=torch.float64, device="cuda")
    # Q = diag(U(1,2)) + U U' with U n x 32 N(0,1)/sqrt(32), "as C2" (SURVEY 8d)
    U = torch.randn((n, 32), generator=g, dtype=torch.float64, device="cuda") / (32 ** 0.5)
    Q = U @ U.t()
    Q.diagonal().add_(qdiag)
    del U
    gs = torch.Generator(device="cuda")
    gs.manual_seed(seed * 7919 + 13)
    s0_full = 0.1 + torch.rand(m, generator=gs, dtype=torch.float64, device="cuda")
    b = At.t() @ y0 - s0_full[r0:r0 + m_loc]
    return dict(name="C4", At=At, b=b, qdiag=qdiag, Q=Q, c=c, cone_dims=[("R", m_loc)], n=n, m=m, m_loc=m_loc)


def _svec(Z):
    """vecm of src/ConicIP.jl:128-151 (row-major upper triangle, off-diagonals * sqrt 2)."""
    k = Z.shape[0]
    iu = np.triu_indices(k)
    x = Z[iu].copy()
    x[iu[0] != iu[1]] *= np.sqrt(2.0)
    return x


def _smat(x):
    """mat of src/ConicIP.jl:93-119."""
    k = int(round((np.sqrt(1 + 8 * len(x)) - 1) / 2))
    Z = np.zeros((k, k))
    iu = np.triu_indices(k)
    Z[iu] = x
    off = iu[0] != iu[1]
    Z[iu[0][off], iu[1][off]] /= np.sqrt(2.0)
    return Z + np.triu(Z, 1).T


def config5(n=20000, k=64, p=1000, seed=5):
    """C5 -- the MOI-shaped LP (Q = 0): x >= 0 on all n variables, one PSD block of order k on the first
    k(k+1)/2 variables, p sparse equality rows (~10 nnz/row); strictly feasible primal and dual by
    construction, so it is bounded (SURVEY 8d).  n = 20000, k = 64, p = 1000 is BASELINE.json's config 5."""
    rng = np.random.default_rng(seed)
    dim = k * (k + 1) // 2
    m = n + dim
    A = np.zeros((m, n))
    A[np.arange(n), np.arange(n)] = 1.0
    A[n + np.arange(dim), np.arange(dim)] = 1.0
    B = rng.standard_normal((k, k)) / np.sqrt(k)
    X0 = B @ B.T + 0.5 * np.eye(k)
    y0 = rng.uniform(0.5, 1.5, n)
    y0[:dim] = np.abs(_svec(X0)) + 0.05            # > 0 entrywise ...
    Xs = _smat(y0[:dim])
    Xs += (0.1 - min(0.0, np.linalg.eigvalsh(Xs).min())) * np.eye(k)      # ... and mat() positive definite
    y0[:dim] = _svec(Xs)
    assert np.linalg.eigvalsh(_smat(y0[:dim])).min() > 0 and y0.min() > 0
    b = np.zeros(m)
    G = np.zeros((p, n))
    for i in range(p):
        G[i, rng.choice(n, min(10, n), replace=False)] = rng.standard_normal(min(10, n))
    d = G @ y0
    v0 = np.zeros(m)
    v0[:n] = rng.uniform(0.5, 1.5, n)
    Bz = rng.standard_normal((k, k)) / np.sqrt(k)
    v0[n:] = _svec(Bz @ Bz.T + 0.5 * np.eye(k))
    w0 = rng.standard_normal(p)
    c = G.T @ w0 - A.T @ v0                          # stationarity (src/ConicIP.jl:747,753): Qy + G'w - A'v = c
    return _prob("C5", np.zeros((n, n)), c, A, b, [("R", n), ("S", dim)], G, d, optTol=1e-8)


def config5_sparse(n=20000, k=64, p=1000, seed=5):
    """C5 built directly in sparse form: A and G as scipy CSC, Q as an empty CSC matrix.  It consumes the same
    random stream as config5, so at equal arguments it is the same problem; it never forms a dense n-wide matrix, so
    it reaches shapes (n = 150 000) where config5's dense A alone would not fit in host memory."""
    rng = np.random.default_rng(seed)
    dim = k * (k + 1) // 2
    m = n + dim
    A = sp.csc_matrix((np.ones(n + dim), (np.arange(m), np.concatenate([np.arange(n), np.arange(dim)]))),
                      shape=(m, n))
    B = rng.standard_normal((k, k)) / np.sqrt(k)
    X0 = B @ B.T + 0.5 * np.eye(k)
    y0 = rng.uniform(0.5, 1.5, n)
    y0[:dim] = np.abs(_svec(X0)) + 0.05
    Xs = _smat(y0[:dim])
    Xs += (0.1 - min(0.0, np.linalg.eigvalsh(Xs).min())) * np.eye(k)
    y0[:dim] = _svec(Xs)
    assert np.linalg.eigvalsh(_smat(y0[:dim])).min() > 0 and y0.min() > 0
    b = np.zeros(m)
    rows, cols, vals = [], [], []
    for i in range(p):
        vals.append(rng.standard_normal(min(10, n)))     # config5's `G[i, choice] = normal` draws the values first
        cols.append(rng.choice(n, min(10, n), replace=False))
        rows.append(np.full(min(10, n), i))
    if p > 0:
        G = sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(p, n))
    else:
        G = sp.csc_matrix((0, n))
    d = G @ y0
    v0 = np.zeros(m)
    v0[:n] = rng.uniform(0.5, 1.5, n)
    Bz = rng.standard_normal((k, k)) / np.sqrt(k)
    v0[n:] = _svec(Bz @ Bz.T + 0.5 * np.eye(k))
    w0 = rng.standard_normal(p)
    c = G.T @ w0 - A.T @ v0
    return _prob("C5", sp.csc_matrix((n, n)), c, A, b, [("R", n), ("S", dim)], G, d, optTol=1e-8)
