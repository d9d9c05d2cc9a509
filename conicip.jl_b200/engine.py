"""`Engine`: thin object wrapper over one `cip_handle` (include/conicip_b200.h).

Vectors may be NumPy arrays (host; results come back as NumPy) or CUDA
`torch.Tensor`s (device; results stay on the device, no PCIe traffic).  PyTorch is
only used to own device memory -- every computation happens in libconicip_b200.so.
"""
import ctypes as C

import numpy as np
import scipy.sparse as sp

from . import _lib
from ._lib import CONE_CODE, Options, Stats, check, lib


def _is_torch(x):
    return hasattr(x, "data_ptr")


def _s_order(dim):
    return int(round((np.sqrt(1 + 8 * dim) - 1) / 2))


def _colmajor(M):
    """Dense column-major float64 (Julia layout) from dense / scipy.sparse / torch input."""
    if M is None:
        return None
    if _is_torch(M):
        return M
    if sp.issparse(M):
        M = M.toarray()
    return np.asfortranarray(M, dtype=np.float64)


class Engine:
    """LEVEL-1 object: `kktsolver(Q, A, G, cone_dims)` (src/ConicIP.jl:667)."""

    def __init__(self, Q, A, G, cone_dims, *, reg_delta=0.0, reg_eps_G=0.0, device=-1,
                 use_torch_stream=True, dist_chol=-1, aug_rho=-1.0, ngpus=1, fold_scaling=0, row_structure=0):
        L = lib()
        self.cone_dims = [(t, int(k)) for t, k in cone_dims]
        self.cone_type = np.array([CONE_CODE[t] for t, _ in self.cone_dims], dtype=np.int32)
        self.cone_dim = np.array([k for _, k in self.cone_dims], dtype=np.int32)
        self.cone_off = np.concatenate([[0], np.cumsum(self.cone_dim)]).astype(np.int64)
        m_c = int(self.cone_off[-1])

        opts = Options()
        opts.struct_size = C.sizeof(Options)
        opts.device = device
        opts.reg_delta = reg_delta
        opts.reg_eps_G = reg_eps_G
        opts.q_kind = 0
        opts.dist_chol = dist_chol
        opts.aug_rho = aug_rho
        opts.ngpus = int(ngpus)            # > 1: single-process multi-GPU handle (global vectors in and out)
        opts.fold_scaling = int(fold_scaling)   # 0 auto, 1 always, 2 never (R-only problems: no Atil copy of A)
        opts.row_structure = int(row_structure)  # 1: singleton R rows on the diagonal, compact SYRK for the rest;
        #                                          2: also factor H as its diagonal plus the coupled block H_KK
        self.ngpus = max(1, int(ngpus))
        self._torch = None
        self._use_torch_stream = use_torch_stream
        self.last_factor_status = 0

        if not _is_torch(A) and sp.issparse(A):
            self._create_csc(Q, A, G, opts)
            return

        # ---- Q: dense, sparse, diagonal vector ("Id(n)", src/ConicIP.jl:18) or None (zero)
        if Q is None:
            opts.q_kind = 2
            q_ptr, ldq, n = None, 0, None
            self._Q = None
        elif not _is_torch(Q) and sp.issparse(Q) and (Q - sp.diags(Q.diagonal())).nnz == 0:
            self._Q = np.ascontiguousarray(Q.diagonal(), dtype=np.float64)
            opts.q_kind = 1
            q_ptr, ldq, n = self._Q.ctypes.data, 1, Q.shape[0]
        else:
            self._Q = _colmajor(Q)
            n = self._Q.shape[0]
            if _is_torch(self._Q):
                # torch is row-major; Q is symmetric so the transpose is the same matrix
                q_ptr, ldq = self._Q.data_ptr(), self._Q.stride(0)
            else:
                q_ptr, ldq = self._Q.ctypes.data, n

        # ---- A: (m x n).  torch input must already be column-major: a (n x m) row-major tensor
        #      passed as `A_colmajor_t` semantics -> we accept A.t() views (stride(0) == 1).
        A = _colmajor(A)
        if _is_torch(A):
            m, nA = A.shape
            if m > 1 and A.stride(0) != 1:
                raise ValueError("device A must be column-major: pass X.t() of a contiguous (n, m) tensor")
            a_ptr, lda = A.data_ptr(), (A.stride(1) if nA > 1 else m)
        else:
            m, nA = A.shape
            a_ptr, lda = (A.ctypes.data if m else None), max(m, 1)
        if n is None:
            n = nA
        if nA != n:
            raise ValueError("Inconsistency in inequalities/objective")
        if m_c != m:
            raise ValueError("cone_dims do not cover the rows of A")

        if G is None:
            p, g_ptr, ldg = 0, None, 1
            self._G = None
        else:
            self._G = _colmajor(G)
            p = self._G.shape[0]
            if self._G.shape[1] != n and p > 0:
                raise ValueError("Inconsistency in equalities/objective")
            if _is_torch(self._G):
                if p > 1 and self._G.stride(0) != 1:
                    raise ValueError("device G must be column-major: pass X.t() of a contiguous (n, p) tensor")
                g_ptr, ldg = self._G.data_ptr(), (self._G.stride(1) if n > 1 else p)
            else:
                g_ptr, ldg = (self._G.ctypes.data if p else None), max(p, 1)

        self.n, self.m, self.p = int(n), int(m), int(p)
        self._h = C.c_void_p()
        rc = L.cip_create(C.byref(self._h), self.n, self.m, self.p, q_ptr, ldq, a_ptr, lda, g_ptr, ldg,
                          len(self.cone_dims), self.cone_type.ctypes.data, self.cone_dim.ctypes.data,
                          C.byref(opts))
        if rc != 0:
            raise _lib.CipError(rc, _lib.last_error())

    def _create_csc(self, Q, A, G, opts):
        """Sparse LEVEL 1 (`cip_create_csc`): CSC arrays go to the device as they are, no dense copy."""
        from ._lib import Csc
        keep = []

        def csc(M):
            if M is None:
                return None
            M = sp.csc_matrix(M, dtype=np.float64)
            M.sum_duplicates()
            cp = np.ascontiguousarray(M.indptr, dtype=np.int64)
            rv = np.ascontiguousarray(M.indices, dtype=np.int64)
            nz = np.ascontiguousarray(M.data, dtype=np.float64)
            keep.extend([cp, rv, nz])
            s = Csc(M.shape[0], M.shape[1], cp.ctypes.data, rv.ctypes.data, nz.ctypes.data, 0)
            keep.append(s)
            return s

        m, n = A.shape
        if Q is not None and Q.shape != (n, n):
            raise ValueError("Inconsistency in inequalities/objective")
        if int(self.cone_off[-1]) != m:
            raise ValueError("cone_dims do not cover the rows of A")
        p = 0 if G is None else G.shape[0]
        if p and G.shape[1] != n:
            raise ValueError("Inconsistency in equalities/objective")
        qs, as_, gs = csc(Q), csc(A), (csc(G) if p else None)
        self.n, self.m, self.p = int(n), int(m), int(p)
        self._h = C.c_void_p()
        rc = lib().cip_create_csc(C.byref(self._h), self.n, C.byref(qs) if qs is not None else None, C.byref(as_),
                                  C.byref(gs) if gs is not None else None, len(self.cone_dims),
                                  self.cone_type.ctypes.data, self.cone_dim.ctypes.data, C.byref(opts))
        if rc != 0:
            raise _lib.CipError(rc, _lib.last_error())

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().cip_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _bind_stream(self):
        if self._torch is None:
            import torch
            self._torch = torch
        if self.ngpus > 1:
            # one stream per device inside the handle: device inputs must be complete before the call
            self._torch.cuda.current_stream().synchronize()
        elif self._use_torch_stream:
            check(lib().cip_set_stream(self._h, self._torch.cuda.current_stream().cuda_stream))

    def _ptr(self, x, length):
        if x is None:
            return None
        if _is_torch(x):
            if not x.is_cuda or x.dtype != self._dtype() or not x.is_contiguous() or x.numel() != length:
                raise ValueError("device vectors must be contiguous CUDA float64 of the right length")
            return x.data_ptr()
        if x.dtype != np.float64 or not x.flags.c_contiguous or x.size != length:
            raise ValueError("host vectors must be contiguous float64 of the right length")
        return x.ctypes.data

    def _dtype(self):
        return self._torch.float64

    def _prep(self, *xs):
        """Normalise inputs; decide whether results live on the device."""
        dev = any(_is_torch(x) for x in xs if x is not None)
        if dev:
            self._bind_stream()
            out = [x if (x is None or _is_torch(x)) else self._torch.as_tensor(np.asarray(x, dtype=np.float64)).cuda()
                   for x in xs]
        else:
            out = [None if x is None else np.ascontiguousarray(x, dtype=np.float64) for x in xs]
        return dev, out

    def _new(self, dev, length):
        if dev:
            return self._torch.empty(length, dtype=self._torch.float64, device="cuda")
        return np.empty(length, dtype=np.float64)

    # ------------------------------------------------------------------ LEVEL 2
    def factor(self, F):
        """`solve3x3gen(F, F^-T)` with a host `Block` (flattened) -- src/ConicIP.jl:682."""
        kind, fa, fb, fD, fR = F.flatten()
        if len(kind) != len(self.cone_dims) or len(fa) != self.m:
            raise ValueError("F does not match cone_dims")
        rc = lib().cip_factor(self._h, kind.ctypes.data, fa.ctypes.data, fb.ctypes.data, fD.ctypes.data,
                              None if fR is None else fR.ctypes.data)
        self.last_factor_status = check(rc)
        return rc

    def factor_resident(self):
        """Form + factor with the scaling already resident (after nt_scaling / set_scaling)."""
        check(lib().cip_form_H(self._h))
        rc = lib().cip_factor_H(self._h)
        self.last_factor_status = check(rc)
        return rc

    def form_H(self):
        check(lib().cip_form_H(self._h))

    def factor_H(self):
        rc = lib().cip_factor_H(self._h)
        self.last_factor_status = check(rc)
        return rc

    def factor_from_point(self, v, s):
        dev, (v, s) = self._prep(v, s)
        lam = self._new(dev, self.m)
        rc = lib().cip_factor_from_point(self._h, self._ptr(v, self.m), self._ptr(s, self.m), self._ptr(lam, self.m))
        self.last_factor_status = check(rc)
        return lam

    def set_scaling(self, F):
        kind, fa, fb, fD, fR = F.flatten()
        check(lib().cip_set_scaling(self._h, kind.ctypes.data, fa.ctypes.data, fb.ctypes.data, fD.ctypes.data,
                                    None if fR is None else fR.ctypes.data))

    def get_scaling(self, with_R=False):
        nc = len(self.cone_dims)
        kind = np.zeros(nc, dtype=np.int32)
        fa, fb, fD = np.zeros(self.m), np.zeros(self.m), np.zeros(nc)
        orders = [_s_order(k) for t, k in self.cone_dims if t == "S"]
        fR = np.zeros(max(1, sum(k * k for k in orders)))
        check(lib().cip_get_scaling(self._h, kind.ctypes.data, fa.ctypes.data, fb.ctypes.data, fD.ctypes.data,
                                    fR.ctypes.data if orders else None))
        if with_R:
            Rs, o = [], 0
            for k in orders:
                Rs.append(fR[o:o + k * k].reshape(k, k, order="F").copy())
                o += k * k
            return kind, fa, fb, fD, Rs
        return kind, fa, fb, fD

    # ------------------------------------------------------------------ LEVEL 3
    def solve(self, ry, rw, rv):
        """`solve3x3(y, w, v) -> (a, b, c)` -- src/kktsolvers.jl:324-332."""
        if rw is None or len(rw) == 0:
            rw = None
        dev, (ry, rw, rv) = self._prep(ry, rw, rv)
        dy, dv = self._new(dev, self.n), self._new(dev, self.m)
        dw = self._new(dev, self.p)
        check(lib().cip_solve(self._h, self._ptr(ry, self.n), self._ptr(rw, self.p) if self.p else None,
                              self._ptr(rv, self.m), self._ptr(dy, self.n),
                              self._ptr(dw, self.p) if self.p else None, self._ptr(dv, self.m)))
        return dy, dw, dv

    def solve_multi(self, RY, RW, RV):
        """`cip_solve_multi`: the columns of RY (n x k), RW (p x k or None), RV (m x k) through the current
        factorisation; A is streamed once per pair of columns.  Column-major (Fortran-ordered NumPy arrays or
        transposed torch tensors) -- column j of the result equals `solve(RY[:, j], RW[:, j], RV[:, j])`."""
        dev = _is_torch(RY) or _is_torch(RV)
        k = int(RY.shape[1])
        if dev:
            self._bind_stream()
            t = self._torch

            def cols(X, rows):            # (rows x k) -> k contiguous columns: a (k, rows) row-major tensor
                if X is None:
                    return None
                X = X if _is_torch(X) else t.as_tensor(np.asarray(X, dtype=np.float64)).cuda()
                Xt = X.t().contiguous()
                assert Xt.shape == (k, rows)
                return Xt
            ry, rw, rv = cols(RY, self.n), cols(RW, self.p) if self.p else None, cols(RV, self.m)
            dy = t.empty((k, self.n), dtype=t.float64, device="cuda")
            dw = t.empty((k, self.p), dtype=t.float64, device="cuda")
            dv = t.empty((k, self.m), dtype=t.float64, device="cuda")
            ptr = lambda x: None if x is None else x.data_ptr()
        else:
            def cols(X, rows):
                if X is None:
                    return None
                Xt = np.ascontiguousarray(np.asarray(X, dtype=np.float64).T)
                assert Xt.shape == (k, rows)
                return Xt
            ry, rw, rv = cols(RY, self.n), cols(RW, self.p) if self.p else None, cols(RV, self.m)
            dy, dw, dv = np.empty((k, self.n)), np.empty((k, self.p)), np.empty((k, self.m))
            ptr = lambda x: None if x is None else x.ctypes.data
        check(lib().cip_solve_multi(self._h, k, ptr(ry), self.n, ptr(rw) if self.p else None, max(self.p, 1),
                                    ptr(rv), self.m, ptr(dy), ptr(dw) if self.p else None, ptr(dv)))
        return dy.T, dw.T, dv.T

    def solve_H(self, rhs):
        """x = inv(H) rhs through the two triangular sweeps alone (`cip_solve_H`, test / bench hook)."""
        dev, (rhs,) = self._prep(rhs)
        x = self._new(dev, self.n)
        check(lib().cip_solve_H(self._h, self._ptr(rhs, self.n), self._ptr(x, self.n)))
        return x

    # ------------------------------------------------------------------ cone kernels
    def nt_scaling(self, v, s):
        dev, (v, s) = self._prep(v, s)
        lam = self._new(dev, self.m)
        rc = check(lib().cip_nt_scaling(self._h, self._ptr(v, self.m), self._ptr(s, self.m), self._ptr(lam, self.m)))
        if rc > 0:      # S-cone iterate not positive definite: PosDefException in the reference (src/ConicIP.jl:201-202)
            raise _lib.CipError(rc, _lib.last_error())
        return lam

    def apply(self, op, x):
        dev, (x,) = self._prep(x)
        y = self._new(dev, self.m)
        check(lib().cip_apply(self._h, op, self._ptr(x, self.m), self._ptr(y, self.m)))
        return y

    def maxstep(self, x, d=None, d_scale=1.0):
        dev, (x, d) = self._prep(x, d)
        a = C.c_double()
        check(lib().cip_maxstep(self._h, self._ptr(x, self.m), self._ptr(d, self.m), float(d_scale), C.byref(a)))
        return a.value

    def cone_prod(self, x, y):
        dev, (x, y) = self._prep(x, y)
        o = self._new(dev, self.m)
        check(lib().cip_cone_prod(self._h, self._ptr(x, self.m), self._ptr(y, self.m), self._ptr(o, self.m)))
        return o

    def cone_div(self, x, y):
        dev, (x, y) = self._prep(x, y)
        o = self._new(dev, self.m)
        check(lib().cip_cone_div(self._h, self._ptr(x, self.m), self._ptr(y, self.m), self._ptr(o, self.m)))
        return o

    # ------------------------------------------------------------------ resident operators
    def mul_A(self, x, trans=False):
        dev, (x,) = self._prep(x)
        nin, nout = (self.m, self.n) if trans else (self.n, self.m)
        y = self._new(dev, nout)
        check(lib().cip_mul_A(self._h, int(trans), self._ptr(x, nin), self._ptr(y, nout)))
        return y

    def mul_G(self, x, trans=False):
        dev, (x,) = self._prep(x)
        nin, nout = (self.p, self.n) if trans else (self.n, self.p)
        y = self._new(dev, nout)
        if nout == 0:
            return y
        check(lib().cip_mul_G(self._h, int(trans), self._ptr(x, nin) if nin else None, self._ptr(y, nout)))
        return y

    def mul_Q(self, x):
        dev, (x,) = self._prep(x)
        y = self._new(dev, self.n)
        check(lib().cip_mul_Q(self._h, self._ptr(x, self.n), self._ptr(y, self.n)))
        return y

    # ------------------------------------------------------------------ native IP loop
    def ipm_solve(self, c, b, d=None, *, optTol=1e-6, DTB=0.01, maxRefinementSteps=3, maxIters=100,
                  infeasTol=None, refinementThreshold=None, verbose=False):
        """`cip_ipm_solve`: the whole of `conicIP` (src/ConicIP.jl:468-939) behind one C call."""
        from ._lib import IpmOptions, IpmResult, STATUS_NAMES
        dev, (c, b, d) = self._prep(c, b, d if (d is not None and len(d)) else None)
        o = IpmOptions()
        o.struct_size = C.sizeof(IpmOptions)
        o.maxIters, o.maxRefinementSteps, o.verbose = int(maxIters), int(maxRefinementSteps), int(verbose)
        o.optTol, o.DTB = float(optTol), float(DTB)
        o.infeasTol = -1.0 if infeasTol is None else float(infeasTol)
        o.refinementThreshold = -1.0 if refinementThreshold is None else float(refinementThreshold)
        y, w, v = self._new(dev, self.n), self._new(dev, self.p), self._new(dev, self.m)
        r = IpmResult()
        check(lib().cip_ipm_solve(self._h, self._ptr(c, self.n), self._ptr(b, self.m) if self.m else None,
                                  self._ptr(d, self.p) if self.p else None, C.byref(o),
                                  self._ptr(y, self.n), self._ptr(w, self.p) if self.p else None,
                                  self._ptr(v, self.m) if self.m else None, C.byref(r)))
        info = {k: getattr(r, k) for k, _ in IpmResult._fields_}
        info["status"] = STATUS_NAMES[r.status]
        return y, w, v, info

    # ------------------------------------------------------------------ multi-GPU / misc
    def comm_init(self, nranks, rank, unique_id):
        check(lib().cip_comm_init(self._h, nranks, rank, unique_id))

    def stats(self):
        st = Stats()
        check(lib().cip_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in Stats._fields_}

    def structure_info(self):
        """How `row_structure=1` split the rows of A (`cip_structure_info`); all zero when the option is off."""
        from ._lib import StructureInfo
        si = StructureInfo()
        si.struct_size = C.sizeof(StructureInfo)
        check(lib().cip_structure_info(self._h, C.byref(si)))
        return {k: getattr(si, k) for k, _ in StructureInfo._fields_ if k != "struct_size"}

    def split_info(self):
        """How `row_structure=2` split the columns of H (`cip_split_info`); all zero otherwise."""
        from ._lib import SplitInfo
        si = SplitInfo()
        si.struct_size = C.sizeof(SplitInfo)
        check(lib().cip_split_info(self._h, C.byref(si)))
        return {k: getattr(si, k) for k, _ in SplitInfo._fields_ if k != "struct_size"}

    def get_H(self):
        out = np.zeros((self.n, self.n), order="F")
        check(lib().cip_get_H(self._h, out.ctypes.data, self.n))
        return out

    def sync(self):
        check(lib().cip_sync(self._h))


def shard_plan(cone_dims, ngpus):
    """Row ranges [(lo, hi)] a handle with `ngpus` devices gives its shards (`cip_shard_plan`, host logic)."""
    ct = np.array([CONE_CODE[t] for t, _ in cone_dims], dtype=np.int32)
    cd = np.array([int(k) for _, k in cone_dims], dtype=np.int32)
    lo, hi = np.zeros(ngpus, dtype=np.int32), np.zeros(ngpus, dtype=np.int32)
    check(lib().cip_shard_plan(len(cd), ct.ctypes.data, cd.ctypes.data, int(ngpus), lo.ctypes.data, hi.ctypes.data))
    return [(int(a), int(b)) for a, b in zip(lo, hi)]


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    check(lib().cip_nccl_unique_id(buf))
    return buf.raw


def measure_fp64_peaks(device=-1):
    a, b = C.c_double(), C.c_double()
    check(lib().cip_measure_fp64_peaks(device, C.byref(a), C.byref(b)))
    return {"dmma_tflops": a.value, "dfma_tflops": b.value}
