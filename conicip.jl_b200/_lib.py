"""ctypes binding of libconicip_b200.so (the C ABI in include/conicip_b200.h).

This is the Python stand-in for the Julia `ccall` shim (julia/ConicIPB200.jl);
both bind exactly the same symbols.  There is NO CPU fallback: if the shared
library is missing or the device is not sm_100a, every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libconicip_b200.so")

CONE_R, CONE_Q, CONE_S = 0, 1, 2
BLK_DIAG, BLK_WOODBURY, BLK_VECCONG = 0, 1, 2
OP_F, OP_FT, OP_FINVT, OP_FINV = 0, 1, 2, 3
CONE_CODE = {"R": CONE_R, "Q": CONE_Q, "S": CONE_S}


class Options(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("device", C.c_int), ("reg_delta", C.c_double),
                ("reg_eps_G", C.c_double), ("q_kind", C.c_int), ("verbose", C.c_int), ("dist_chol", C.c_int), ("aug_rho", C.c_double),
                ("ngpus", C.c_int), ("fold_scaling", C.c_int), ("row_structure", C.c_int)]


class StructureInfo(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("enabled", C.c_int), ("singleton_rows", C.c_int), ("empty_rows", C.c_int),
                ("rest_rows", C.c_int), ("rest_cols", C.c_int), ("compressed", C.c_int), ("base_has_gtg", C.c_int)]


class SplitInfo(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("enabled", C.c_int), ("coupled_cols", C.c_int), ("diagonal_cols", C.c_int),
                ("cols_from_rest", C.c_int), ("cols_from_Q", C.c_int), ("cols_from_G", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("n", C.c_int), ("m", C.c_int), ("p", C.c_int),
                ("n_pad", C.c_int), ("m_pad", C.c_int), ("p_pad", C.c_int),
                ("factors", C.c_longlong), ("solves", C.c_longlong),
                ("ms_scale", C.c_double), ("ms_syrk", C.c_double), ("ms_allreduce", C.c_double),
                ("ms_chol", C.c_double), ("ms_schur", C.c_double), ("ms_solve", C.c_double),
                ("syrk_flops", C.c_double), ("chol_flops", C.c_double),
                ("device_bytes", C.c_size_t), ("kernel_launches", C.c_longlong)]


class Csc(C.Structure):
    _fields_ = [("nrows", C.c_int), ("ncols", C.c_int), ("colptr", C.c_void_p), ("rowval", C.c_void_p),
                ("nzval", C.c_void_p), ("index_base", C.c_int)]


class IpmOptions(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("maxIters", C.c_int), ("maxRefinementSteps", C.c_int), ("verbose", C.c_int),
                ("optTol", C.c_double), ("DTB", C.c_double), ("infeasTol", C.c_double),
                ("refinementThreshold", C.c_double)]


class IpmResult(C.Structure):
    _fields_ = [("status", C.c_int), ("Iter", C.c_int), ("factors", C.c_int), ("solves", C.c_int),
                ("Mu", C.c_double), ("prFeas", C.c_double), ("duFeas", C.c_double), ("muFeas", C.c_double),
                ("pobj", C.c_double), ("dobj", C.c_double), ("seconds", C.c_double)]


STATUS_NAMES = {0: "None", 1: "Optimal", 2: "Infeasible", 3: "Unbounded", 4: "Abandoned", 5: "Error"}


class CipError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"conicip_b200 error {code}: {msg}")
        self.code = code


_lib = None
_P = C.c_void_p   # every double*/int* argument: host or device address

# name -> (restype, argtypes); mirrors include/conicip_b200.h line by line
SIGNATURES = {
    "cip_last_error": (C.c_char_p, []),
    "cip_version": (C.c_int, []),
    "cip_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int,
                             _P, C.c_int, C.c_int, _P, _P, C.POINTER(Options)]),
    "cip_create_csc": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(Csc), C.POINTER(Csc), C.POINTER(Csc),
                                 C.c_int, _P, _P, C.POINTER(Options)]),
    "cip_destroy": (C.c_int, [C.c_void_p]),
    "cip_shard_plan": (C.c_int, [C.c_int, _P, _P, C.c_int, _P, _P]),
    "cip_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "cip_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "cip_factor": (C.c_int, [C.c_void_p, _P, _P, _P, _P, _P]),
    "cip_factor_from_point": (C.c_int, [C.c_void_p, _P, _P, _P]),
    "cip_solve": (C.c_int, [C.c_void_p, _P, _P, _P, _P, _P, _P]),
    "cip_solve_multi": (C.c_int, [C.c_void_p, C.c_int, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "cip_nt_scaling": (C.c_int, [C.c_void_p, _P, _P, _P]),
    "cip_get_scaling": (C.c_int, [C.c_void_p, _P, _P, _P, _P, _P]),
    "cip_set_scaling": (C.c_int, [C.c_void_p, _P, _P, _P, _P, _P]),
    "cip_apply": (C.c_int, [C.c_void_p, C.c_int, _P, _P]),
    "cip_maxstep": (C.c_int, [C.c_void_p, _P, _P, C.c_double, C.POINTER(C.c_double)]),
    "cip_cone_prod": (C.c_int, [C.c_void_p, _P, _P, _P]),
    "cip_cone_div": (C.c_int, [C.c_void_p, _P, _P, _P]),
    "cip_mul_A": (C.c_int, [C.c_void_p, C.c_int, _P, _P]),
    "cip_mul_G": (C.c_int, [C.c_void_p, C.c_int, _P, _P]),
    "cip_mul_Q": (C.c_int, [C.c_void_p, _P, _P]),
    "cip_ipm_solve": (C.c_int, [C.c_void_p, _P, _P, _P, C.POINTER(IpmOptions), _P, _P, _P, C.POINTER(IpmResult)]),
    "cip_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "cip_structure_info": (C.c_int, [C.c_void_p, C.POINTER(StructureInfo)]),
    "cip_split_info": (C.c_int, [C.c_void_p, C.POINTER(SplitInfo)]),
    "cip_get_H": (C.c_int, [C.c_void_p, _P, C.c_int]),
    "cip_form_H": (C.c_int, [C.c_void_p]),
    "cip_factor_H": (C.c_int, [C.c_void_p]),
    "cip_solve_H": (C.c_int, [C.c_void_p, _P, _P]),
    "cip_sync": (C.c_int, [C.c_void_p]),
    "cip_stream": (C.c_void_p, [C.c_void_p]),
    "cip_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cip_measure_fp64_peaks": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "cip_imcols": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p,
                             C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C conicip.jl_b200/csrc).  conicip_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code < 0:
        raise CipError(code, lib().cip_last_error().decode())
    return code


def last_error():
    return lib().cip_last_error().decode()
