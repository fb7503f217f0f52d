"""ctypes binding of libqmpc.so (include/qmpc.h).  PyTorch tensors provide device memory; this module only
passes their data_ptr()s through the C-ABI.  There is no CPU fallback: if the CUDA library is missing or was
not built, loading raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QMPC_LIB", os.path.join(_HERE, "csrc", "libqmpc.so"))   # QMPC_LIB: kernel-tuning experiments only
_LIB = None

NX, NU, NY = 13, 4, 17


class QmpcConfig(C.Structure):
    """mirror of `qmpc_config` (include/qmpc.h)"""
    _fields_ = [
        ("batch", C.c_int), ("n_nodes", C.c_int), ("n_basis", C.c_int), ("precision", C.c_int),
        ("device", C.c_int), ("ipm_max_iter", C.c_int), ("refine_max_rounds", C.c_int), ("warm_start_rounds", C.c_int),
        ("ipm_mu_tol", C.c_double), ("ipm_mu_switch", C.c_double), ("t_horizon", C.c_double),
        ("quad", C.c_double * 20), ("w_diag", C.c_double * 17), ("we_diag", C.c_double * 13),
        ("lbu", C.c_double), ("ubu", C.c_double), ("gp_theta", C.c_double * 9),
        ("gp_X", C.POINTER(C.c_double)),
        ("solver_variant", C.c_int), ("reset_on_fail", C.c_int), ("screen_rounds", C.c_int), ("dense_warm_rounds", C.c_int),
        ("bail_round", C.c_int), ("bail_changed", C.c_int), ("final_rollout", C.c_int), ("dense_grid", C.c_int),
        ("screen_rounds_busy", C.c_int), ("screen_busy_pct", C.c_int),
    ]


class QmpcError(RuntimeError):
    pass


def lib():
    """Load libqmpc.so; raises (never falls back) if it is absent."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise QmpcError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). mpc_quad_ros_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.qmpc_last_error.restype = C.c_char_p
        L.qmpc_launch_count.restype = C.c_longlong
        L.qrgp_Kx_inv_device.restype = C.c_void_p
        L.qrgp_mu_device.restype = C.c_void_p
        L.qmpc_eval_jvp.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise QmpcError(f"libqmpc error {rc}: {lib().qmpc_last_error().decode()}")


def ptr(t):
    """device pointer of a contiguous CUDA tensor (or NULL)"""
    if t is None:
        return C.c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "libqmpc takes contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)
