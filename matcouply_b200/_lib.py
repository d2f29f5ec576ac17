"""ctypes binding of the C ABI declared in ``include/matcouply_b200.h`` (``libmatcouply_b200.so``).

There is NO CPU fallback: if the shared library is missing, or a call fails, this module raises.
The library has no torch dependency; torch is only used by the callers for device memory and streams.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2_LIB_PATH_DEBUG") or os.path.join(_HERE, "libmatcouply_b200.so")

F32, F64 = 0, 1
VARIANT_AUTO, VARIANT_FMA, VARIANT_DMMA = 0, 1, 2
PEN_NONNEG, PEN_BOX, PEN_L1, PEN_L2BALL, PEN_UNIMODAL, PEN_PARAFAC2, PEN_GL2, PEN_SIMPLEX, PEN_TV, PEN_HOST = range(10)
PEN_TEMPORAL = 10
GROUP_SINGLE, GROUP_INDEXED, GROUP_IDENTITY = 0, 1, 2
OPT_PF2_ROWPASS_MMA, OPT_POLAR_WARP, OPT_ADMM_LOCAL_MMA, OPT_XSTREAM_HYBRID, OPT_UNIMODAL_VARIANT = 0, 1, 2, 3, 4
# B2_OPT_PF2_ROWPASS_MMA: 0 = shuffle kernel, 1 = DMMA tile kernel, 2 (default) = + the steady-state specialisation
PF2_ROWPASS_DEFAULT = 2
MAX_RANK = 32
MAX_PENALTIES_PER_MODE = 4


class PenaltyDesc(ctypes.Structure):
    """Mirror of ``b2_penalty_desc``."""

    _fields_ = [
        ("kind", ctypes.c_int32),
        ("non_negativity", ctypes.c_int32),
        ("p0", ctypes.c_double),
        ("p1", ctypes.c_double),
        ("aux", ctypes.c_void_p),
        ("dual", ctypes.c_void_p),
    ]


_vp, _i, _ll, _sz, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_size_t, ctypes.c_double

# name -> argtypes ; every function returns int status except the ones listed in _OTHER_RESTYPE
_SIGNATURES = {
    "b2_xstream_y": [_vp, _ll, _i, _i, _vp, _i, _vp, _i, _vp, _sz, _i, _i, _vp],
    "b2_xstream_z": [_vp, _ll, _i, _i, _vp, _i, _i, _vp, _i, _vp, _sz, _i, _i, _vp],
    "b2_sumsq": [_vp, _ll, _i, _i, _i, _vp, _vp, _sz, _vp],
    "b2_xstream_fused_local": [_vp, _ll, _i, _i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, ctypes.POINTER(PenaltyDesc),
                               _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp],
    "b2_slice_gdot": [_vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "b2_gram": [_vp, _ll, _i, _i, _vp, _i, _vp, _sz, _vp],
    "b2_scale_gram": [_vp, _vp, _i, _i, _vp, _i, _vp],
    "b2_rho_from_trace": [_vp, _i, _i, _d, _vp, _vp, _i, _vp],
    "b2_factor_batch": [_vp, _i, _i, _vp, _vp, _i, _d, _vp, _i, _vp],
    "b2_slice_cross": [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp],
    "b2_rowscale": [_vp, _vp, _vp, _ll, _i, _vp, _i, _i, _vp],
    "b2_admm_solve": [_ll, _i, _vp, _vp, _i, _vp, _vp, _vp, ctypes.POINTER(PenaltyDesc), _i, _vp, _i, _vp],
    "b2_admm_local": [_ll, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, ctypes.POINTER(PenaltyDesc), _i, _i, _vp, _vp, _i,
                      _vp, _i, _vp],
    "b2_prox_l2ball": [_vp, _vp, _vp, _i, _i, _d, _i, _vp, _i, _i, _vp],
    "b2_prox_unimodal": [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _sz, _vp],
    "b2_selftest_div_count": [_ll, ctypes.c_ulonglong, _i, _vp, _vp],
    "b2_prox_simplex": [_vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "b2_prox_tv": [_vp, _vp, _vp, _i, _i, _vp, _i, _d, _d, _i, _vp],
    "b2_tv_norm": [_vp, _vp, _i, _i, _vp, _vp, _i, _vp],
    "b2_prox_gl2": [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _i, _vp],
    "b2_quadform": [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp],
    "b2_pf2_fixed_basis": [_vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _vp, _vp, _i, _i, _vp],
    "b2_pf2_polar": [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp],
    "b2_pf2_rowpass": [_vp, _i, _i, _vp, _vp, _vp, _vp, ctypes.POINTER(PenaltyDesc), _i, _i, _vp, _vp, _vp, _vp, _i, _vp,
                       _vp, _vp, _i, _vp],
    "b2_group_stats_sum": [_vp, _i, _vp, _vp],
    "b2_pf2_delta": [_vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp],
    "b2_pf2_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp],
    "b2_pf2_gap": [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp, _sz, _vp],
    "b2_slice_gram": [_vp, _vp, _i, _i, _vp, _i, _vp],
    "b2_slice_coldot": [_vp, _vp, _vp, _i, _i, _vp, _i, _vp],
    "b2_weighted_gram_sum": [_vp, _vp, _i, _i, _vp, _i, _vp],
    "b2_hadamard_bcast": [_vp, _vp, _i, _i, _vp, _i, _vp],
    "b2_reduce_stats": [_vp, _vp, _ll, _vp, _i, _vp, _sz, _vp],
    "b2_fit_terms": [_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _sz, _vp],
    "b2_prox_elementwise": [_vp, _vp, _ll, _i, _i, _d, _d, _d, _i, _vp],
    "b2_microbench_flops": [_i, _i, ctypes.POINTER(_d), _vp, _vp],
    "b2_mt19937_uniform": [_vp, _vp, _ll, _vp],
    "b2_mt19937_jump_host": [_vp, ctypes.c_ulonglong],
    "b2_set_option": [_i, _i],
    "b2_mask_refill": [_vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp, _sz, _vp],
    "b2_prox_temporal": [_vp, _vp, _ll, _ll, _vp, _i, _d, _i, _i, _i, _vp, _i, _i, _i, _vp, _sz, _vp],
    "b2_prox_temporal_serial": [_vp, _vp, _ll, _ll, _vp, _i, _d, _i, _vp, _sz, _vp],
    "b2_temporal_norm": [_vp, _ll, _ll, _d, _vp, _i, _vp, _vp, _i, _vp],
}
_OTHER = {
    "b2_last_error": ([], ctypes.c_char_p),
    "b2_version": ([], _i),
    "b2_device_sm_count": ([], _i),
    "b2_launch_count": ([], ctypes.c_ulonglong),
    "b2_get_option": ([_i], _i),
    "b2_pf2_rowpass_fused_stats_supported": ([_i, _i, _i, _i, _i], _i),
    "b2_xstream_workspace_bytes": ([_i, _i, _i], _sz),
    "b2_xstream_fused_local_supported": ([_i, _i, _i, _i], _i),
    "b2_xstream_fused_workspace_bytes": ([_i, _i, _i], _sz),
    "b2_xstream_z_ldw": ([_i, _i, _i], _i),
    "b2_unimodal_workspace_bytes": ([_i, _i, _i], _sz),
    "b2_mask_refill_workspace_bytes": ([_ll], _sz),
    "b2_prox_temporal_workspace_bytes": ([_ll, _ll, _i], _sz),
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + list(_OTHER))

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """Load the shared library (once). Raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C matcouply_b200/csrc`). matcouply_b200 has no CPU fallback."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, args in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _i
        for name, (args, res) in _OTHER.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = res
        _lib = lib
    return _lib


def call(name, *args):
    """Invoke a status-returning entry point and raise on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.b2_last_error()
        raise RuntimeError(f"{name} failed (status {rc}): {msg.decode() if msg else '?'}")


def dtype_code(torch_dtype):
    import torch

    if torch_dtype == torch.float64:
        return F64
    if torch_dtype == torch.float32:
        return F32
    raise TypeError(f"matcouply_b200 supports float32 and float64, not {torch_dtype}")
