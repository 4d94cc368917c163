"""ctypes binding of libprmf_b200.so (include/prmf_b200.h).  No torch types cross this boundary."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint8, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libprmf_b200.so")

OBJ_STRIDE = 8
UNIQUE_ID_BYTES = 128
IPC_HANDLE_BYTES = 64
N_PHASES = 6
X_DTYPES = {"f64": 0, "tf32": 1, "f32": 2}          # PRMF_X_F64 / PRMF_X_TF32 / PRMF_X_F32
PHASES = ("xv", "u_update", "xtu", "reduce", "v_update", "objective")

# every symbol include/prmf_b200.h declares: name -> (restype, argtypes)
_P = c_void_p
SYMBOLS = {
    "prmf_abi_version": (c_int, []),
    "prmf_create": (c_int, [POINTER(_P), c_int, c_int64, c_int64, c_int64, c_int, _P]),
    "prmf_create_ex": (c_int, [POINTER(_P), c_int, c_int64, c_int64, c_int64, c_int, _P, c_int]),
    "prmf_x_dtype": (c_int, [_P]),
    "prmf_destroy": (c_int, [_P]),
    "prmf_last_error": (c_char_p, [_P]),
    "prmf_set_X": (c_int, [_P, _P, c_int64]),
    "prmf_set_X_device": (c_int, [_P, _P, c_int64]),
    "prmf_set_X_f32": (c_int, [_P, _P, c_int64, c_int]),
    "prmf_get_normX_sq": (c_int, [_P, POINTER(c_double)]),
    "prmf_set_pathways": (c_int, [_P, c_int32, _P, _P, _P, _P, _P]),
    "prmf_set_UV": (c_int, [_P, _P, _P]),
    "prmf_get_UV": (c_int, [_P, _P, _P]),
    "prmf_set_active": (c_int, [_P, _P]),
    "prmf_step": (c_int, [_P, c_int, c_double, c_double, c_double, _P, _P]),
    "prmf_step_async": (c_int, [_P, c_int, c_double, c_double, c_double]),
    "prmf_step_collect": (c_int, [_P, c_int, _P, _P]),
    "prmf_scores": (c_int, [_P, _P, _P, _P]),
    "prmf_block_end": (c_int, [_P, c_int, _P, _P, c_int, _P, _P, _P, c_int]),
    "prmf_snapshot_best": (c_int, [_P]),
    "prmf_restore_best": (c_int, [_P]),
    "prmf_residual_sq": (c_int, [_P, POINTER(c_double)]),
    "prmf_objective": (c_int, [_P, c_double, c_double, _P]),
    "prmf_nccl_load": (c_int, [c_char_p]),
    "prmf_comm_unique_id": (c_int, [POINTER(c_uint8)]),
    "prmf_comm_init": (c_int, [_P, c_int, c_int, POINTER(c_uint8)]),
    "prmf_p2p_export": (c_int, [_P, POINTER(c_uint8)]),
    "prmf_p2p_attach": (c_int, [_P, c_int, c_int, POINTER(c_uint8)]),
    "prmf_p2p_finalize": (c_int, [_P]),
    "prmf_exchange_mode": (c_int, [_P]),
    "prmf_launch_count": (c_int64, [_P]),
    "prmf_kernel_times": (c_int, [_P, c_int, POINTER(c_double), POINTER(c_int64)]),
    "prmf_set_profiling": (c_int, [_P, c_int]),
    "prmf_project": (c_int, [_P, _P]),
    "prmf_project_t": (c_int, [_P, _P]),
    "prmf_nnls_x": (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P]),
    "prmf_release_pool": (c_int, []),
    "prmf_debug_inject_fault": (c_int, [_P, c_int]),
    "prmf_stream": (_P, [_P]),
    "prmf_quantile_transform": (c_int, [c_int, _P, _P, c_int64, c_int64, c_int64, _P, c_int64, c_int, _P, _P, _P, _P, _P,
                                        c_int64, _P]),
    "prmf_preprocess_last_error": (c_char_p, []),
    "prmf_nnls_rows": (c_int, [c_int, _P, c_int64, c_int, _P, c_int64, c_int64, _P, _P, _P, _P]),
    "prmf_cv_last_error": (c_char_p, []),
    "prmf_host_restrict": (c_int64, [_P, _P, _P, c_int64, c_double, _P, _P]),
    "prmf_host_restrict_batch": (c_int64, [_P, _P, c_int64, c_int32, _P, _P, _P, c_double, _P, _P, _P]),
}

_lib = None


class PrmfLibraryError(RuntimeError):
    pass


def load(build_if_missing=True):
    """Load the shared library.  It is built in-tree by `prmf_b200.build` (nvcc, sm_100a); a missing
    library is an error -- there is no other execution path."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from . import build
        try:
            if build.is_stale():
                build.build_library()
        except Exception as exc:  # nvcc absent on the GPU box is fine as long as the .so travelled
            if not os.path.exists(LIB_PATH):
                raise PrmfLibraryError("libprmf_b200.so is missing and could not be built: %s" % exc)
    if not os.path.exists(LIB_PATH):
        raise PrmfLibraryError("libprmf_b200.so not found at %s (run `python -m prmf_b200.build`)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(lib, handle, rc):
    if rc != 0:
        msg = lib.prmf_last_error(handle)
        raise PrmfLibraryError("libprmf_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
