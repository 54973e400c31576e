"""ctypes binding of libdifflinker_b200.so (include/difflinker_b200.h). No CPU fallback: if the library or a
B200 is missing, calls fail loudly."""
import ctypes as C
import os

from .build import LIB_PATH, build_native, is_stale, nvcc_path

DL_OK, DL_NAN_DETECTED = 0, 1
GRAPH_TYPES = {"FC": 0, "4A": 1, "FC-4A": 2, "FC-10A-4A": 3}
EDGE_IMPLS = {"auto": 0, "simt": 1, "tcgen05": 2}
SAMPLER_LINKER, SAMPLER_INPAINT = 0, 1
# dl_diffusion_loss: rows of the per-molecule coefficient table and columns of the per-molecule terms
LOSS_COEFS = ("t", "alpha_t", "sigma_t", "alpha_1", "sigma2_1", "log_inv_sigma_1")
LOSS_TERMS = ("error_t", "noise", "log_p_x", "log_p_h", "kl_prior", "n_linker")


class DLConfig(C.Structure):
    _fields_ = [("n_dims", C.c_int32), ("in_node_nf", C.c_int32), ("context_node_nf", C.c_int32),
                ("hidden_nf", C.c_int32), ("n_layers", C.c_int32), ("inv_sublayers", C.c_int32),
                ("condition_time", C.c_int32), ("centering", C.c_int32), ("graph_type", C.c_int32),
                ("device", C.c_int32), ("edge_impl", C.c_int32), ("norm_constant", C.c_float),
                ("normalization_factor", C.c_float)]


class DLSizeGNNConfig(C.Structure):
    _fields_ = [("in_node_nf", C.c_int32), ("hidden_nf", C.c_int32), ("out_node_nf", C.c_int32),
                ("n_layers", C.c_int32), ("device", C.c_int32)]


class DLStepCoef(C.Structure):
    _fields_ = [("t", C.c_float), ("a", C.c_float), ("b", C.c_float), ("c", C.c_float), ("frame", C.c_int32),
                ("qa", C.c_float), ("qb", C.c_float), ("pad", C.c_float)]


# every symbol include/difflinker_b200.h declares: name -> (restype, argtypes)
_P, _I32, _I64, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SYMBOLS = {
    "dl_version": (C.c_char_p, []),
    "dl_last_error": (C.c_char_p, []),
    "dl_create": (_I32, [C.POINTER(DLConfig), C.POINTER(_P)]),
    "dl_destroy": (_I32, [_P]),
    "dl_set_weight": (_I32, [_P, C.c_char_p, _P, _I64]),
    "dl_finalize_weights": (_I32, [_P]),
    "dl_expected_param_count": (_I64, [_P]),
    "dl_dynamics_forward": (_I32, [_P, _I32, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dl_dynamics_forward_host": (_I32, [_P, _I32, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "dl_sample_chain": (_I32, [_P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dl_sample_chain_rng": (_I32, [_P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, C.c_uint64, C.c_uint64, _P, _P, _P, _P,
                                   _P, _P]),
    "dl_diffusion_loss": (_I32, [_P, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, C.c_uint64, C.c_uint64, _P, _P, _P, _P, _P]),
    "dl_set_noise_slice": (_I32, [_P, _I32, _I32]),
    "dl_noise_fill": (_I32, [_P, _I32, _I32, _I32, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "dl_sample_chain_host": (_I32, [_P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dl_launch_count": (_I64, [_P]),
    "dl_last_elapsed_ms": (_F, [_P]),
    "dl_time_edge_kernel": (_F, [_P, _I32]),
    "dl_selftest_tc": (_I32, [_P, C.POINTER(_F), C.POINTER(_F)]),
    "dl_selftest_tc_layout": (_I32, [_P, _I32, C.POINTER(_F), C.POINTER(_F)]),
    "dl_cut_graph_stats": (_I32, [_P, C.POINTER(_I64)]),
    "dl_sizegnn_create": (_I32, [C.POINTER(DLSizeGNNConfig), C.POINTER(_P)]),
    "dl_sizegnn_destroy": (_I32, [_P]),
    "dl_sizegnn_set_weight": (_I32, [_P, C.c_char_p, _P, _I64]),
    "dl_sizegnn_finalize_weights": (_I32, [_P]),
    "dl_sizegnn_forward": (_I32, [_P, _I32, _I32, _P, _P, _P, _P, _P]),
    "dl_restore_frame": (_I32, [_I32, _I32, _I32, _P, _P, _P, _P, _P]),
    "dl_restore_frame2": (_I32, [_I32, _I32, _I32, _I32, _P, _P, _P, _P, _P]),
    "dl_bond_orders": (_I32, [_I32, _I32, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "dl_format_xyz": (_I64, [_I32, _I32, _I32, _P, _I32, _P, _I32, _P, C.POINTER(C.c_char_p), _I32, _P, _I64, _P]),
}

_lib = None


def load_library():
    """Loads (building first when stale and nvcc is around) the native library. Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if is_stale():
        if nvcc_path() is not None:
            build_native()
        elif not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing and nvcc is unavailable; build it with `python -m difflinker_b200.build`. "
                "difflinker_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class NativeError(RuntimeError):
    pass


def check(status: int, what: str):
    if status < 0:
        raise NativeError(f"{what} failed with status {status}: {load_library().dl_last_error().decode()}")
    return status
