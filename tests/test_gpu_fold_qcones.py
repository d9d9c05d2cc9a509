"""fold_scaling with second-order cones: the SYRK forms F^-T A row by row from At4 and the cones' T rows (no Atil4).

H is checked elementwise against an FP64 reference built from the oracle's own NT scaling blocks (the bound of
tests/test_gpu_row_structure_reference.py), against the materialised handle, and end to end through cip_ipm_solve.
The cone layouts put many cones in one 32-row k tile (dimension 3: sixteen slots), cones that straddle tile edges
(31, 32, 33), one cone across many tiles (1500 rows) and R rows between the cones.
"""
import numpy as np
import pytest

import oracle as O
from conicip_b200 import problems as P
from test_gpu_row_structure_reference import assert_H, cone_point, oracle_F, ref_H

KNOBS = ("CIP_FOLD_SCALING", "CIP_ROW_STRUCTURE", "CIP_FAST_SYRK")

LAYOUTS = {
    "dim3": [("Q", 3)] * 70,
    "dim33": [("R", 4)] + [("Q", 33)] * 12,
    "dim31": [("R", 5)] + [("Q", 31)] * 12,
    "dim32": [("R", 7)] + [("Q", 32)] * 12,
    "dim1500": [("R", 20), ("Q", 1500), ("R", 13)],
    "mixed": [("R", 10), ("Q", 33), ("R", 3), ("Q", 5), ("R", 40), ("Q", 33), ("R", 1), ("Q", 7), ("Q", 3)] * 3,
}


@pytest.fixture(autouse=True)
def _option_decides(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def make(cones, n=300, p=0, seed=0):
    rng = np.random.default_rng(seed)
    m = sum(k for _, k in cones)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    G = rng.standard_normal((p, n)) / np.sqrt(n) if p else None
    Q = P._lowrank_q(rng, n, 8)
    return Q, A, G


def engines(Q, A, G, cones, **kw):
    import conicip_b200 as cb
    return (cb.Engine(Q, A, G, cones, fold_scaling=1, **kw), cb.Engine(Q, A, G, cones, fold_scaling=2, **kw))


def H_at(e, v, s):
    e.nt_scaling(v, s)
    e.form_H()
    return e.get_H()


def rho_of(p, aug_rho=-1.0):
    return (aug_rho if aug_rho >= 0 else 1.0) if p > 0 else 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_folded_H_against_fp64_reference(layout):
    cones = LAYOUTS[layout]
    Q, A, G = make(cones, seed=len(layout))
    ef, em = engines(Q, A, G, cones)
    rng = np.random.default_rng(3)
    m, n = A.shape
    m_pad, n_pad = (m + 31) // 32 * 32, (n + 127) // 128 * 128
    # no second copy of A: the folded handle holds at least m_pad x n_pad doubles less, less its T rows
    drop = em.stats()["device_bytes"] - ef.stats()["device_bytes"]
    assert drop >= m_pad * n_pad * 8 * 0.45, drop
    for wide in (True, False):
        v, s = cone_point(cones, rng, wide), cone_point(cones, rng, wide)
        ref = ref_H(Q, A, G, cones, oracle_F(cones, v, s), 0.0)
        Hf, Hm = H_at(ef, v, s), H_at(em, v, s)
        assert_H(Hf, ref, f"{layout} folded {'wide' if wide else 'central'}")
        assert_H(Hm, ref, f"{layout} materialised {'wide' if wide else 'central'}")


@pytest.mark.gpu
@pytest.mark.parametrize("aug_rho", [-1.0, 0.0])
def test_folded_equality_block(aug_rho):
    cones = LAYOUTS["mixed"]
    Q, A, G = make(cones, p=7, seed=5)
    ef, em = engines(Q, A, G, cones, aug_rho=aug_rho)
    rng = np.random.default_rng(4)
    v, s = cone_point(cones, rng), cone_point(cones, rng)
    ref = ref_H(Q, A, G, cones, oracle_F(cones, v, s), rho_of(G.shape[0], aug_rho))
    assert_H(H_at(ef, v, s), ref, f"folded aug_rho={aug_rho}")
    assert_H(H_at(em, v, s), ref, f"materialised aug_rho={aug_rho}")
    # and the KKT solves agree
    for e in (ef, em):
        e.factor_from_point(v, s)
    ry, rw, rv = rng.standard_normal(A.shape[1]), rng.standard_normal(G.shape[0]), rng.standard_normal(A.shape[0])
    for a, b in zip(ef.solve(ry, rw, rv), em.solve(ry, rw, rv)):
        assert rel(a, b) < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["dim3", "dim33", "dim1500", "mixed"])
def test_folded_against_materialised(layout):
    """H, its Cholesky factor L, cip_solve and cip_solve_multi of the folded handle against the materialised one"""
    cones = LAYOUTS[layout]
    Q, A, G = make(cones, p=4, seed=11)
    ef, em = engines(Q, A, G, cones)
    rng = np.random.default_rng(8)
    v, s = cone_point(cones, rng), cone_point(cones, rng)
    ref = ref_H(Q, A, G, cones, oracle_F(cones, v, s), 1.0)
    tol = 4 * 2.0 ** -53 * (ref.k + 2) * ref.B
    Hf, Hm = H_at(ef, v, s), H_at(em, v, s)
    lower = np.tril_indices(A.shape[1])
    assert np.all((np.abs(Hf - Hm) <= 2 * tol)[lower])
    for e in (ef, em):
        e.factor_from_point(v, s)
    Lf, Lm = np.tril(ef.get_H()), np.tril(em.get_H())
    assert rel(Lf, Lm) < 1e-12
    n, m, p = A.shape[1], A.shape[0], G.shape[0]
    ry, rw, rv = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(m)
    for a, b in zip(ef.solve(ry, rw, rv), em.solve(ry, rw, rv)):
        assert rel(a, b) < 1e-10
    RY, RW, RV = (np.asfortranarray(rng.standard_normal(sh)) for sh in ((n, 3), (p, 3), (m, 3)))
    for a, b in zip(ef.solve_multi(RY, RW, RV), em.solve_multi(RY, RW, RV)):
        assert rel(a, b) < 1e-10


@pytest.mark.gpu
def test_initial_diag_call_is_the_r_formula():
    """F = I on every block (the first call of conicIP, DIAG blocks in the Q slots): H = Q + A'A"""
    import conicip_b200 as cb
    cones = LAYOUTS["mixed"]
    Q, A, G = make(cones, seed=2)
    ef, _ = engines(Q, A, G, cones)
    # any diagonal F (the identity first): the Q slots behave as R rows
    for d in (np.ones(A.shape[0]), np.random.default_rng(1).uniform(0.2, 5.0, A.shape[0])):
        blocks, oblocks, off = [], [], 0
        for _, k in cones:
            blocks.append(cb.Diagonal(d[off:off + k]))
            oblocks.append(O.Diag(d[off:off + k]))
            off += k
        ef.set_scaling(cb.Block(blocks))
        ef.form_H()
        assert_H(ef.get_H(), ref_H(Q, A, G, cones, O.Block(oblocks), 0.0), "diagonal F")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["dim3", "mixed"])
def test_folded_H_is_deterministic(layout):
    cones = LAYOUTS[layout]
    Q, A, G = make(cones, seed=9)
    ef, _ = engines(Q, A, G, cones)
    rng = np.random.default_rng(6)
    v, s = cone_point(cones, rng), cone_point(cones, rng)
    H1 = H_at(ef, v, s)
    H2 = H_at(ef, v, s)
    assert np.array_equal(H1.view(np.uint64), H2.view(np.uint64))


# sha256 of tril(H) of the folded K = R^m handle below, formed by the R-only instance (W^-2 on the Y fragments) on one
# B200 (148 SMs: the split-K plan of the SYRK depends on the SM count)
R_FOLD_H_SHA256 = "33e014ed4b8c02b8bc5eba50ca4135452b5ae7d71ef92c7f637566105ef6a574"


@pytest.mark.gpu
def test_r_only_fold_unchanged():
    """K = R^m keeps the R-only instance: its H is bit for bit the stored one, reproducible from call to call, within
    the reference bound; the handle holds no T rows"""
    import hashlib
    import torch
    import conicip_b200 as cb
    rng = np.random.default_rng(12)
    m, n = 700, 300
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    Q = P._lowrank_q(rng, n, 8)
    cones = [("R", m)]
    ef = cb.Engine(Q, A, None, cones, fold_scaling=1)
    em = cb.Engine(Q, A, None, cones, fold_scaling=2)
    m_pad, n_pad = (m + 31) // 32 * 32, (n + 127) // 128 * 128
    assert em.stats()["device_bytes"] - ef.stats()["device_bytes"] == m_pad * n_pad * 8
    v, s = cone_point(cones, rng, True), cone_point(cones, rng, True)
    H1, H2 = H_at(ef, v, s), H_at(ef, v, s)
    assert np.array_equal(H1.view(np.uint64), H2.view(np.uint64))
    assert_H(H1, ref_H(Q, A, None, cones, oracle_F(cones, v, s), 0.0), "R fold")
    if torch.cuda.get_device_properties(0).multi_processor_count == 148:
        assert hashlib.sha256(np.ascontiguousarray(np.tril(H1)).tobytes()).hexdigest() == R_FOLD_H_SHA256


def oracle_solve(prob):
    return O.conicIP(prob["Q"], prob["c"], prob["A"], prob["b"], prob["cone_dims"], prob["G"], prob["d"],
                     kktsolver=O.pivot(O.kktsolver_2x2), optTol=1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C3_reduced", "soc_equalities"])
def test_folded_full_solve_against_oracle(name):
    import conicip_b200 as cb
    prob = P.config3(n=512, ncones=64, k=33, p=32) if name == "C3_reduced" else P.mixed(n=200, mr=60, ncones=20, k=33, p=9)
    so = oracle_solve(prob)
    G = prob["G"] if prob["G"].shape[0] else None
    e = cb.Engine(prob["Q"], prob["A"], G, prob["cone_dims"], fold_scaling=1)
    em = cb.Engine(prob["Q"], prob["A"], G, prob["cone_dims"], fold_scaling=2)
    assert e.stats()["device_bytes"] < em.stats()["device_bytes"]
    y, w, v, info = e.ipm_solve(prob["c"], prob["b"], prob["d"], optTol=1e-8)
    assert info["status"] == so.status == "Optimal"
    assert abs(info["Iter"] - so.Iter) <= 1
    assert rel(y, so.y) < 1e-6 and rel(w, so.w) < 1e-6 and rel(v, so.v) < 1e-6


@pytest.mark.gpu
def test_sharded_folded_matches_single_device():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    import conicip_b200 as cb
    cones = LAYOUTS["mixed"] * 2
    Q, A, G = make(cones, p=5, seed=13)
    e1 = cb.Engine(Q, A, G, cones, fold_scaling=1)
    e2 = cb.Engine(Q, A, G, cones, fold_scaling=1, ngpus=2)
    rng = np.random.default_rng(14)
    v, s = cone_point(cones, rng), cone_point(cones, rng)
    H1, H2 = H_at(e1, v, s), H_at(e2, v, s)
    ref = ref_H(Q, A, G, cones, oracle_F(cones, v, s), 1.0)
    assert_H(H1, ref, "single device")
    assert_H(H2, ref, "sharded")


@pytest.mark.gpu
def test_auto_keeps_a_fitting_qcone_handle_materialised():
    """fold_scaling = 0 folds an R + Q problem only when the second copy of A would not fit: a small one keeps
    Atil4 and forms the same H, bit for bit, as fold_scaling = 2"""
    import conicip_b200 as cb
    cones = LAYOUTS["mixed"]
    Q, A, G = make(cones, p=3, seed=15)
    ea = cb.Engine(Q, A, G, cones, fold_scaling=0)
    em = cb.Engine(Q, A, G, cones, fold_scaling=2)
    assert ea.stats()["device_bytes"] == em.stats()["device_bytes"]
    rng = np.random.default_rng(16)
    v, s = cone_point(cones, rng), cone_point(cones, rng)
    assert np.array_equal(H_at(ea, v, s).view(np.uint64), H_at(em, v, s).view(np.uint64))


@pytest.mark.gpu
def test_folded_H_at_scale():
    """A tall A (m = 33 * 6000 rows): the slot table must reach the device after the zero fill of a large At4
    and every k tile must still find its cones' T rows"""
    cones = [("R", 11)] + [("Q", 33)] * 6000
    rng = np.random.default_rng(17)
    n = 512
    A = rng.standard_normal((sum(k for _, k in cones), n)) / np.sqrt(n)
    Q = np.eye(n)
    ef, em = engines(Q, A, None, cones)
    for wide in (False, True):
        v, s = cone_point(cones, rng, wide), cone_point(cones, rng, wide)
        Hf, Hm = H_at(ef, v, s), H_at(em, v, s)
        lower = np.tril_indices(n)
        assert np.array_equal(Hf[lower].view(np.uint64), Hm[lower].view(np.uint64)) or \
            rel(Hf[lower], Hm[lower]) < 1e-13
