"""ctypes binding of libmaxent_b200.so (the C ABI declared in include/maxent_b200.h).

There is NO fallback: if the shared library is missing the import of anything that computes raises
``MaxEntLibraryError`` telling the user to run ``python -m maxent_b200.build``.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# MAXENT_B200_LIB selects another build of the same library (A/B timing of kernel variants, tools/ab_bench.py)
LIB_PATH = os.environ.get("MAXENT_B200_LIB") or os.path.join(HERE, "libmaxent_b200.so")

MX_OK = 0
MX_MAX_NSV = 256
MX_MAX_MATRIX = 8
VARIANTS = {"normal": 0, "plusminus": 1, "bryan": 2}
AN_LINEFIT, AN_CHI2CURV, AN_ENTROPY, AN_CLASSIC, AN_BRYAN = range(5)
N_ANALYZERS = 5
STATUS_CONVERGED = 1
STATUS_SKIPPED = 2
PER_SPECTRUM_MODEL, PER_SPECTRUM_XI, PER_SPECTRUM_VT, PER_SPECTRUM_ALPHA = 1, 2, 4, 8
_ERR = {-1: "bad argument", -2: "unsupported (n_sv too large for the fused path?)", -3: "CUDA error",
        -4: "no CUDA device"}

c_dp = ctypes.c_void_p


class MaxEntLibraryError(RuntimeError):
    pass


class MxLMParams(ctypes.Structure):
    _fields_ = [("maxiter", ctypes.c_int32), ("miniter", ctypes.c_int32), ("mu0", ctypes.c_double),
                ("nu", ctypes.c_double), ("max_mu", ctypes.c_double),
                ("conv_max_derivative", ctypes.c_double), ("conv_rel_change", ctypes.c_double),
                ("conv_abs_change", ctypes.c_double), ("marquardt", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class MxProblem(ctypes.Structure):
    _fields_ = [("n_tau", ctypes.c_int32), ("n_omega", ctypes.c_int32), ("n_sv", ctypes.c_int32),
                ("n_alpha", ctypes.c_int32), ("variant", ctypes.c_int32), ("want_probability", ctypes.c_int32),
                ("per_spectrum_model", ctypes.c_int32), ("chi2_factor", ctypes.c_double),
                ("Vt", c_dp), ("Qw", c_dp), ("Qo", c_dp), ("sqrtw", c_dp), ("xi", c_dp), ("D", c_dp),
                ("delta", c_dp), ("alpha", c_dp), ("v0", c_dp), ("lm", MxLMParams), ("vt_index", c_dp),
                ("vt_stride", ctypes.c_int64)]


class MxSweepOut(ctypes.Structure):
    _fields_ = [("v", c_dp), ("A", c_dp), ("chi2", c_dp), ("S", c_dp), ("Q", c_dp), ("logp", c_dp),
                ("n_iter", c_dp), ("n_qeval", c_dp), ("n_solve", c_dp), ("status", c_dp),
                ("n_trial", c_dp), ("n_batch", c_dp), ("phase_cycles", c_dp)]


# every symbol include/maxent_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("mx_version", ctypes.c_char_p, []),
    ("mx_device_sm_count", ctypes.c_int, []),
    ("mx_fp64_peak", ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), c_dp, c_dp]),
    ("mx_layout_V_size", ctypes.c_int64, [ctypes.c_int32, ctypes.c_int32]),
    ("mx_layout_V", ctypes.c_int, [c_dp, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp]),
    ("mx_tau_kernel", ctypes.c_int, [c_dp, c_dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, c_dp, c_dp]),
    ("mx_iomega_kernel", ctypes.c_int, [c_dp, c_dp, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp]),
    ("mx_svd_jacobi", ctypes.c_int, [c_dp, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp, c_dp, c_dp,
                                     ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), c_dp]),
    ("mx_gram_schmidt_rows", ctypes.c_int, [c_dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.c_void_p]),
    ("mx_svd_truncated_work_doubles", ctypes.c_int64, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
    ("mx_svd_truncated", ctypes.c_int, [c_dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp, c_dp, c_dp,
                                        ctypes.c_uint64, c_dp]),
    ("mx_project_data", ctypes.c_int, [ctypes.POINTER(MxProblem), c_dp, ctypes.c_int32, c_dp, c_dp, c_dp]),
    ("mx_alpha_sweep", ctypes.c_int, [ctypes.POINTER(MxProblem), c_dp, c_dp, ctypes.c_int32,
                                      ctypes.POINTER(MxSweepOut), c_dp, ctypes.c_int64, c_dp]),
    ("mx_sweep_workspace_bytes", ctypes.c_int64, [ctypes.POINTER(MxProblem), ctypes.c_int32]),
    ("mx_sweep_config", ctypes.c_int, [ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    ("mx_analyze", ctypes.c_int, [c_dp, c_dp, c_dp, c_dp, c_dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                  ctypes.c_double, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp, c_dp, c_dp]),
    ("mx_poorman_models", ctypes.c_int, [c_dp, ctypes.c_int32, c_dp, ctypes.c_int32, c_dp, ctypes.c_double, c_dp, c_dp,
                                         c_dp, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp, c_dp, c_dp]),
    ("mx_hilbert_table", ctypes.c_int, [c_dp, ctypes.c_int32, c_dp, ctypes.c_int32, ctypes.c_double, c_dp, c_dp]),
    ("mx_hilbert_apply", ctypes.c_int, [c_dp, ctypes.c_int64, ctypes.c_int32, c_dp, ctypes.c_int32, ctypes.c_int32, c_dp,
                                        ctypes.c_double, ctypes.c_int32, c_dp, c_dp, c_dp, c_dp]),
    ("mx_matrix_resolvent", ctypes.c_int, [c_dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, c_dp, c_dp, ctypes.c_int32,
                                           c_dp, c_dp]),
]

_lib = None


def load():
    """Load the shared library (once) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MaxEntLibraryError(
            "libmaxent_b200.so not found at %s -- build it with `python -m maxent_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc, what):
    if rc != MX_OK:
        raise MaxEntLibraryError("%s failed: %s (code %d)" % (what, _ERR.get(rc, "unknown"), rc))


def sweep_config(n_sv):
    lib = load()
    sm, th = ctypes.c_int32(), ctypes.c_int32()
    check(lib.mx_sweep_config(n_sv, ctypes.byref(sm), ctypes.byref(th)), "mx_sweep_config")
    return dict(smem_bytes=sm.value, threads=th.value)
