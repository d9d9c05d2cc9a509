"""`conicIP`: host driver with the reference's signature, running on the B200 engine.

A transliteration of /root/reference/src/ConicIP.jl:468-939 (Mehrotra predictor-corrector
with Nesterov-Todd scaling) in which every O(m), O(mn) and O(n^3) operation is a call into
libconicip_b200.so on device-resident vectors (`Engine`): the KKT levels (:667,:682,:688),
`nt_scaling` (:589), `maxstep` (:571), `cone_prod!`/`cone_div!` (:622-665), the block applies
and the residual mat-vecs (:747-750,:912-914).  Only control flow and scalar arithmetic run
here -- the part that stays in Julia in a ConicIP.jl deployment (julia/ConicIPB200.jl).

Row-sharded multi-GPU: pass `reducer=` (see dist.py); m-vectors are then this rank's slab and
scalar reductions over m go through it.
"""
import math
from dataclasses import dataclass, field

import numpy as np

from ._lib import OP_F, OP_FINVT, OP_FT
from .blocks import Block, DeviceBlock, Diagonal
from .kktsolver import kktsolver_b200


@dataclass
class Solution:
    """src/ConicIP.jl:384-398."""
    y: np.ndarray
    w: np.ndarray
    v: np.ndarray
    status: str = "None"
    Iter: int = 0
    Mu: float = 0.0
    prFeas: float = math.inf
    duFeas: float = math.inf
    muFeas: float = math.inf
    pobj: float = math.inf
    dobj: float = -math.inf
    trace: list = field(default_factory=list)
    solves: int = 0
    factors: int = 0


class _V4:
    __slots__ = ("y", "w", "v", "s")

    def __init__(self, y, w, v, s):
        self.y, self.w, self.v, self.s = y, w, v, s


class LocalReducer:
    """Single-GPU: reductions over m are local."""
    nranks = 1

    def sum(self, x):
        return x

    def min(self, x):
        return x

    def sum_tensor_(self, t):
        return t

    def min_list(self, xs):
        return list(xs)


def conicIP_native(Q, c, A, b, cone_dims, G=None, d=None, *, engine=None, ngpus=1, row_structure=0, **opts):
    """Same problem statement and options as `conicIP`, but the loop itself runs inside the library
    (`cip_ipm_solve`, SURVEY 8f rank 1): one C call per solve.  Pass `engine=` to reuse a handle;
    `ngpus > 1` row-shards A over that many devices of this process (`cip_options.ngpus`);
    `row_structure=1` exploits the row structure of A when forming H (`cip_options.row_structure`);
    `row_structure=2` also factors H as its diagonal plus the coupled block, with no n x n buffer."""
    from .engine import Engine
    eng = engine or Engine(Q, A, G if (G is not None and G.shape[0]) else None, cone_dims, ngpus=ngpus,
                           row_structure=row_structure)
    y, w, v, info = eng.ipm_solve(np.asarray(c, dtype=np.float64), np.asarray(b, dtype=np.float64),
                                  None if d is None else np.asarray(d, dtype=np.float64), **opts)
    sol = Solution(np.asarray(y), np.asarray(w), np.asarray(v), status=info["status"], Iter=info["Iter"],
                   Mu=info["Mu"], prFeas=info["prFeas"], duFeas=info["duFeas"], muFeas=info["muFeas"],
                   pobj=info["pobj"], dobj=info["dobj"], solves=info["solves"], factors=info["factors"])
    sol.seconds = info["seconds"]
    if engine is None:
        eng.close()
    return sol


def conicIP(Q, c, A, b, cone_dims, G=None, d=None, *, kktsolver=kktsolver_b200,
            optTol=1e-6, DTB=0.01, verbose=False, maxRefinementSteps=3, maxIters=100,
            infeasTol=None, refinementThreshold=None, reducer=None, global_cone_dims=None):
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("conicip_b200.conicIP needs a CUDA (sm_100a) device; there is no CPU path")
    R = reducer or LocalReducer()
    dev = torch.device("cuda")
    f64 = torch.float64

    def T(x):
        return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).to(dev)

    c_h = np.asarray(c, dtype=np.float64)
    b_h = np.asarray(b, dtype=np.float64)
    n = len(c_h)
    d_h = np.zeros(0) if d is None else np.asarray(d, dtype=np.float64)
    infeasTol = optTol if infeasTol is None else infeasTol
    refinementThreshold = optTol / 1e7 if refinementThreshold is None else refinementThreshold

    m = A.shape[0]
    p = 0 if G is None else G.shape[0]
    # sanity checks, src/ConicIP.jl:536-542
    if Q is not None and Q.shape[0] != Q.shape[1]:
        raise ValueError("Q is not square")
    if b_h.shape[0] != m:
        raise ValueError("Inconsistency in inequalities")
    if A.shape[1] != n or (Q is not None and Q.shape[0] != n):
        raise ValueError("Inconsistency in inequalities/objective")
    if d_h.shape[0] != p:
        raise ValueError("Inconsistency in equalities")
    if G is not None and p > 0 and G.shape[1] != n:
        raise ValueError("Inconsistency in equalities/objective")

    block_types = [t for t, _ in cone_dims]
    block_sizes = [int(k) for _, k in cone_dims]
    offs = np.concatenate([[0], np.cumsum(block_sizes)]).astype(int)
    # conedim / e, src/ConicIP.jl:547-565 (conedim is global under sharding)
    e_h = np.zeros(m)
    conedim = 0
    for t, k, o in zip(block_types, block_sizes, offs[:-1]):
        if t == "R":
            conedim += k
            e_h[o:o + k] = 1.0
        elif t == "Q":
            conedim += 1
            e_h[o] = 1.0
        else:                                    # S: vecm(I), src/ConicIP.jl:551,564
            ks = int(round((math.sqrt(1 + 8 * k) - 1) / 2))
            conedim += ks
            idx, pos = 0, []
            for i in range(ks):
                pos.append(o + idx)
                idx += ks - i
            e_h[pos] = 1.0
    conedim = int(round(R.sum(float(conedim))))

    c_t, b_t, d_t, e_t = T(c_h), T(b_h), T(d_h), T(e_h)

    zero = torch.zeros((), dtype=f64, device=dev)
    m_glob = int(round(R.sum(float(m))))

    def dots(local_pairs, shard_pairs=()):
        """All the inner products of one phase with ONE host synchronisation: `local_pairs` are
        replicated n-/p-vectors, `shard_pairs` are m-vectors whose partial sums are all-reduced
        across the row shards (one small collective) before the single device->host read."""
        vals = [torch.dot(x, y) if x.numel() else zero for x, y in local_pairs]
        nl = len(vals)
        vals += [torch.dot(x, y) if x.numel() else zero for x, y in shard_pairs]
        t = torch.stack(vals)
        if len(shard_pairs):
            R.sum_tensor_(t[nl:])
        out = t.tolist()
        return out[:nl], out[nl:]

    def nrm(x):
        return float(torch.linalg.vector_norm(x).item()) if x.numel() else 0.0

    def mnrm(x):
        return math.sqrt(dots((), ((x, x),))[1][0])

    normc = nrm(c_t)
    normd = -math.inf if p == 0 else nrm(d_t)
    normb = mnrm(b_t)

    solve3x3gen = kktsolver(Q, A, G, cone_dims)                      # :667  LEVEL 1
    eng = solve3x3gen.engine

    def maxstep2(x1, d1, x2, d2, scale=1.0):                         # :571-587, two calls, one reduction
        return R.min_list([eng.maxstep(x1, d1, scale), eng.maxstep(x2, d2, scale)])

    counters = {"solves": 0, "factors": 0}

    def solve4x4gen(lam, F, Finvt):                                  # :669-694
        counters["factors"] += 1
        solve3x3 = solve3x3gen(F, Finvt)                             # LEVEL 2

        def solve4x4(r):
            counters["solves"] += 1
            t1 = eng.apply(OP_FT, eng.cone_div(r.s, lam))
            dy, dw, dv = solve3x3(r.y, r.w, r.v + t1)                # LEVEL 3
            if not torch.is_tensor(dy):                              # failed factorisation -> NaNs
                dy, dw, dv = T(dy), T(dw), T(dv)
            t1 = t1 - eng.apply(OP_FT, eng.apply(OP_F, dv))
            return _V4(dy, dw, dv, t1)

        return solve4x4

    # ---- initial point :704-713 (F = I: Diagonal blocks for every cone, Q slots included)
    I0 = Block([Diagonal(np.ones(k)) for k in block_sizes])
    r0 = _V4(c_t, d_t, b_t, torch.zeros(m, dtype=f64, device=dev))
    z = solve4x4gen(e_t, I0, I0)(r0)
    a_v, a_s = maxstep2(z.v, None, z.s, None)
    z.v = z.v - a_v * e_t
    z.s = z.s - a_s * e_t

    sol = Solution(None, None, None)
    optBest = math.inf
    nan = math.nan

    def finish(status, y=None, w=None, v=None):
        sol.status = status
        sol.y = (z.y if y is None else y).cpu().numpy()
        sol.w = (z.w if w is None else w).cpu().numpy()
        sol.v = (z.v if v is None else v).cpu().numpy()
        sol.solves, sol.factors = counters["solves"], counters["factors"]
        return sol

    for Iter in range(1, maxIters + 1):                              # :730
        lam = eng.nt_scaling(z.v, z.s)                               # F resident on the device
        F = DeviceBlock(eng)
        Finvt = DeviceBlock(eng, inverse_adjoint=True)
        solve = solve4x4gen(lam, F, Finvt)

        Qy = eng.mul_Q(z.y)
        Gtw = eng.mul_G(z.w, trans=True)
        Atv = eng.mul_A(z.v, trans=True)
        Ay = eng.mul_A(z.y)
        rleft = _V4(Qy + Gtw - Atv, eng.mul_G(z.y), Ay - z.s, eng.cone_prod(lam, lam))
        r0 = _V4(rleft.y - c_t, rleft.w - d_t, rleft.v - b_t, rleft.s)   # :753

        gtw_atv = Gtw - Atv
        ay_s = Ay - z.s
        (cty, r0y2, yQy, w_r0w, dtw, gta2, yy, gy2, qy2), (mubar, r0v2, r0s2, v_r0v, btv, vv, ays2) = dots(
            ((c_t, z.y), (r0.y, r0.y), (z.y, Qy), (z.w, r0.w), (d_t, z.w), (gtw_atv, gtw_atv), (z.y, z.y),
             (rleft.w, rleft.w), (Qy, Qy)),
            ((z.v, z.s), (r0.v, r0.v), (r0.s, r0.s), (z.v, r0.v), (b_t, z.v), (z.v, z.v), (ay_s, ay_s)))
        mu = mubar / conedim
        rDu = math.sqrt(r0y2) / (1 + normc)
        rPr = math.sqrt(r0v2) / (1 + normb)
        rCp = math.sqrt(r0s2) / (1 + abs(cty))
        sol.trace.append((Iter, mu, rDu, rPr, rCp))

        if max(rDu, rPr, rCp) < optBest:                             # :768-773
            sol.Iter, sol.Mu = Iter, mu
            sol.duFeas, sol.prFeas, sol.muFeas = rDu, rPr, rCp
            optBest = max(rDu, rPr, rCp)

        pobj = 0.5 * yQy - cty
        dobj = pobj + w_r0w + v_r0v - mubar
        sol.pobj, sol.dobj = pobj, dobj

        status = "None"
        out_y = out_w = out_v = None
        if max(rDu, rPr, rCp) < optTol:                              # :786
            status = "Optimal"

        if not (p == 0 and m == 0):                                  # :790-852
            dty_btv = dtw - btv
            p_unscaled = math.sqrt(gta2)
            if dty_btv < 0:
                with np.errstate(all="ignore"):
                    p_cvx = np.float64(p_unscaled) / (math.sqrt(yy) + math.sqrt(vv))
                    p_ecos = np.float64(p_unscaled) / (max(1, normc) * abs(dty_btv))
            else:
                p_cvx = p_ecos = nan
            p_infeas = float(np.maximum(p_cvx, p_ecos))
            if p_infeas < infeasTol:
                out_y = torch.full_like(z.y, nan)
                out_w = z.w / -dty_btv
                out_v = z.v / -dty_btv
                status = "Infeasible"

            d1 = -math.inf if m_glob == 0 else math.sqrt(ays2)
            d2 = -math.inf if p == 0 else math.sqrt(gy2)
            d3 = math.sqrt(qy2) if math.isfinite(yy) else nan
            if cty > 0:
                d_cvx = max(d1 / max(1, normb), d2 / max(1, normd), d3 / max(1, normc)) / abs(cty)
                d_ecos = max(d1, d2, d3) / math.sqrt(yy)
            else:
                d_cvx = d_ecos = nan
            d_infeas = abs(float(np.maximum(d_cvx, d_ecos)))
            if d_infeas < infeasTol:
                out_y = z.y / abs(cty)
                out_v = torch.full_like(z.v, nan)
                out_w = torch.full_like(z.w, nan)
                status = "Unbounded"

        if verbose:
            print(f" {Iter:6d}  | {rDu:8.1e} {rPr:8.1e} {rCp:8.1e} | {pobj: 8.1e} {dobj: 8.1e} | mu {mu:8.1e}",
                  flush=True)

        if status != "None":
            return finish(status, out_y, out_w, out_v)
        if not all(math.isfinite(t) for t in (mu, rDu, rPr, rCp)):   # :870-873
            return finish("Error")

        # ---- predictor :879-887
        d_aff = solve(r0)
        a1, a2 = maxstep2(z.v, d_aff.v, z.s, d_aff.s)
        a_aff = min(min(a1, 1), min(a2, 1))
        # fts(), :162-163
        _, (v_ds, dv_s, dv_ds) = dots((), ((z.v, d_aff.s), (d_aff.v, z.s), (d_aff.v, d_aff.s)))
        rho = (mubar - a_aff * v_ds - a_aff * dv_s + a_aff * a_aff * dv_ds) / mubar
        sigma = max(0, min(1, rho)) ** 3

        # ---- corrector :893-901
        lc = eng.cone_prod(eng.apply(OP_FINVT, d_aff.s), eng.apply(OP_F, d_aff.v))
        lc = -(lc - (sigma * mu) * e_t)
        r = _V4(r0.y, r0.w, r0.v, rleft.s - lc)

        # ---- newton step + iterative refinement :907-921
        dz = solve(r)
        for _ in range(maxRefinementSteps):
            pb1 = eng.cone_prod(lam, eng.apply(OP_F, dz.v))
            pb2 = eng.cone_prod(lam, eng.apply(OP_FINVT, dz.s))
            rI = _V4(r.y - (eng.mul_Q(dz.y) + eng.mul_G(dz.w, trans=True) - eng.mul_A(dz.v, trans=True)),
                     r.w - eng.mul_G(dz.y),
                     r.v - (eng.mul_A(dz.y) - dz.s),
                     r.s - (pb1 + pb2))
            (ry2, rw2), (rv2, rs2) = dots(((rI.y, rI.y), (rI.w, rI.w)), ((rI.v, rI.v), (rI.s, rI.s)))
            rnorm = (math.sqrt(ry2) + math.sqrt(rw2) + math.sqrt(rv2) + math.sqrt(rs2)) / (n + 2 * m_glob)
            if rnorm < refinementThreshold:
                break
            dzr = solve(rI)
            dz.y += dzr.y
            dz.w += dzr.w
            dz.v += dzr.v
            dz.s += dzr.s

        # ---- step :927-932
        a_v, a_s = maxstep2(z.v, dz.v, z.s, dz.s, 1 - DTB)
        alpha = min(min(a_v, 1), min(a_s, 1))
        z.y = z.y - alpha * dz.y
        z.w = z.w - alpha * dz.w
        z.v = z.v - alpha * dz.v
        z.s = z.s - alpha * dz.s

    return finish("Abandoned")
