"""ctypes binding of csrc/libsiren_b200.so (C ABI: include/siren_b200.h).

The library is built in-tree (``make -C siren_mri_b200/csrc`` or ``__graft_entry__.build()``).
Loading fails loudly: the native path has no silent fallback.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libsiren_b200.so")

PREC_FP32 = 0
PREC_BF16 = 1
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16}

# every symbol include/siren_b200.h declares
SYMBOLS = [
    "siren_b200_version", "siren_b200_last_error", "siren_b200_device_ok", "siren_b200_workspace_bytes",
    "siren_b200_workspace_bytes_ex",
    "siren_b200_forward", "siren_b200_forward_infer", "siren_b200_backward", "siren_b200_adam", "siren_b200_mse_grad",
    "siren_b200_forward_ff", "siren_b200_backward_ff",
    "siren_b200_forward_dc", "siren_b200_backward_dc", "siren_b200_forward_dc_mse",
    "siren_b200_hyper_head", "siren_b200_forward_call", "siren_b200_backward_call",
    "siren_b200_publish", "siren_b200_prepare_weights", "siren_b200_forward_prepared", "siren_b200_forward_mse",
    "siren_b200_forward_backward_mse",
    "siren_b200_adam_step", "siren_b200_adam_step_peers", "siren_b200_clip_grad", "siren_b200_loss_roll",
    "siren_b200_adam_step_tasks", "siren_b200_clip_grad_tasks",
    "siren_b200_laplace_mse_grad", "siren_b200_sdf_grad",
    "siren_b200_debug_linear", "siren_b200_debug_wgrad", "siren_b200_profile_begin", "siren_b200_profile_end",
    "siren_b200_comm_unique_id", "siren_b200_comm_init", "siren_b200_allreduce", "siren_b200_comm_destroy",
    "siren_b200_comm_last_error", "siren_b200_allreduce_peers", "siren_b200_allreduce_multicast",
]


class SirenDesc(ctypes.Structure):
    _fields_ = [
        ("d_in", ctypes.c_int), ("hidden", ctypes.c_int), ("n_hidden", ctypes.c_int), ("d_out", ctypes.c_int),
        ("w0", ctypes.c_float), ("tasks", ctypes.c_int), ("per_task", ctypes.c_int),
        ("n_coords", ctypes.c_long), ("precision", ctypes.c_int), ("deriv_order", ctypes.c_int),
    ]


class SirenFourier(ctypes.Structure):      # siren_fourier_t (include/siren_b200.h)
    _fields_ = [("B", ctypes.c_void_p), ("n_features", ctypes.c_int), ("raw_dim", ctypes.c_int)]


class SirenDC(ctypes.Structure):           # siren_dc_t (include/siren_b200.h)
    _fields_ = [("k0", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("noise_lvl", ctypes.c_float),
                ("channels_first", ctypes.c_int)]


class SirenCall(ctypes.Structure):         # siren_call_t (include/siren_b200.h)
    _fields_ = [("fourier", ctypes.POINTER(SirenFourier)), ("dc", ctypes.POINTER(SirenDC)),
                ("wk16", ctypes.POINTER(ctypes.c_void_p)), ("wt16", ctypes.POINTER(ctypes.c_void_p))]


class NativeError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()


def _bind(lib):
    vp, fp, ci, cl, cf = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_float
    cd = ctypes.c_double
    pd = ctypes.POINTER(SirenDesc)
    pp = ctypes.POINTER(ctypes.c_void_p)
    lib.siren_b200_version.restype = ci
    lib.siren_b200_last_error.restype = ctypes.c_char_p
    lib.siren_b200_device_ok.restype = ci
    lib.siren_b200_workspace_bytes.restype = ctypes.c_size_t
    lib.siren_b200_workspace_bytes.argtypes = [pd]
    lib.siren_b200_workspace_bytes_ex.restype = ctypes.c_size_t
    lib.siren_b200_workspace_bytes_ex.argtypes = [pd, ci]
    lib.siren_b200_forward.restype = ci
    lib.siren_b200_forward.argtypes = [pd, fp, pp, pp, fp, fp, fp, vp, vp]
    lib.siren_b200_forward_infer.restype = ci
    lib.siren_b200_forward_infer.argtypes = [pd, fp, pp, pp, fp, vp, vp]
    lib.siren_b200_backward.restype = ci
    lib.siren_b200_backward.argtypes = [pd, fp, pp, pp, vp, fp, fp, fp, pp, pp, fp, ci, vp]
    pf = ctypes.POINTER(SirenFourier)
    lib.siren_b200_forward_ff.restype = ci
    lib.siren_b200_forward_ff.argtypes = [pd, pf, fp, pp, pp, fp, vp, ci, vp]
    lib.siren_b200_backward_ff.restype = ci
    lib.siren_b200_backward_ff.argtypes = [pd, pf, fp, pp, pp, vp, fp, pp, pp, ci, vp]
    pc = ctypes.POINTER(SirenDC)
    lib.siren_b200_forward_dc.restype = ci
    lib.siren_b200_forward_dc.argtypes = [pd, pf, pc, fp, pp, pp, fp, vp, ci, vp]
    lib.siren_b200_backward_dc.restype = ci
    lib.siren_b200_backward_dc.argtypes = [pd, pf, pc, fp, pp, pp, vp, fp, pp, pp, ci, vp]
    lib.siren_b200_forward_dc_mse.restype = ci
    lib.siren_b200_forward_dc_mse.argtypes = [pd, pf, pc, fp, pp, pp, fp, fp, cf, fp, fp, vp, vp]
    pk = ctypes.POINTER(SirenCall)
    lib.siren_b200_hyper_head.restype = ci
    lib.siren_b200_hyper_head.argtypes = [fp, fp, fp, ci, ci, cf, fp, vp, vp, fp, vp]
    lib.siren_b200_forward_call.restype = ci
    lib.siren_b200_forward_call.argtypes = [pd, pk, fp, pp, pp, fp, vp, ci, vp]
    lib.siren_b200_backward_call.restype = ci
    lib.siren_b200_backward_call.argtypes = [pd, pk, fp, pp, pp, vp, fp, pp, pp, ci, vp]
    lib.siren_b200_adam.restype = ci
    lib.siren_b200_adam.argtypes = [fp, fp, fp, fp, cl, cf, cd, cd, cf, cf, cf, vp, vp]
    lib.siren_b200_prepare_weights.restype = ci
    lib.siren_b200_prepare_weights.argtypes = [pd, pp, vp, vp]
    lib.siren_b200_forward_prepared.restype = ci
    lib.siren_b200_forward_prepared.argtypes = [pd, fp, pp, pp, fp, fp, fp, vp, vp]
    lib.siren_b200_forward_mse.restype = ci
    lib.siren_b200_forward_mse.argtypes = [pd, fp, pp, pp, fp, fp, cf, fp, fp, vp, ci, vp]
    lib.siren_b200_forward_backward_mse.restype = ci
    lib.siren_b200_forward_backward_mse.argtypes = [pd, fp, pp, pp, fp, fp, cf, fp, fp, vp, ci, pp, pp, ci, vp]
    lib.siren_b200_adam_step.restype = ci
    lib.siren_b200_adam_step.argtypes = [fp, fp, fp, fp, cl, cf, cd, cd, cf, cf, cf, vp, ci, fp, pd, pp, vp, vp]
    lib.siren_b200_laplace_mse_grad.restype = ci
    lib.siren_b200_laplace_mse_grad.argtypes = [fp, fp, fp, cl, ci, cf, fp, vp]
    lib.siren_b200_sdf_grad.restype = ci
    lib.siren_b200_sdf_grad.argtypes = [fp, fp, fp, fp, fp, fp, cl, cf, fp, vp]
    lib.siren_b200_adam_step_peers.restype = ci
    lib.siren_b200_adam_step_peers.argtypes = [fp, fp, fp, fp, cl, cf, cd, cd, cf, cf, cf, vp, fp, pd, pp, vp, vp, ci, fp, vp]
    lib.siren_b200_clip_grad.restype = ci
    lib.siren_b200_clip_grad.argtypes = [fp, cl, cf, vp, vp]
    lib.siren_b200_adam_step_tasks.restype = ci
    lib.siren_b200_adam_step_tasks.argtypes = [pd, pp, pp, fp, fp, fp, fp, cl, cf, cd, cd, cf, cf, vp, fp, fp, cf, fp, fp,
                                               fp, vp, vp]
    lib.siren_b200_clip_grad_tasks.restype = ci
    lib.siren_b200_clip_grad_tasks.argtypes = [pd, pp, pp, fp, cl, cf, vp, fp, fp, cf, fp, fp, fp, ci, vp]
    lib.siren_b200_loss_roll.restype = ci
    lib.siren_b200_loss_roll.argtypes = [fp, vp]
    lib.siren_b200_mse_grad.restype = ci
    lib.siren_b200_mse_grad.argtypes = [fp, fp, fp, cl, cf, fp, vp]
    lib.siren_b200_publish.restype = ci
    lib.siren_b200_publish.argtypes = [fp, vp, ci, vp]
    lib.siren_b200_profile_begin.restype = ci
    lib.siren_b200_profile_end.restype = ci
    lib.siren_b200_profile_end.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    lib.siren_b200_comm_unique_id.restype = ci
    lib.siren_b200_comm_unique_id.argtypes = [vp]
    lib.siren_b200_comm_init.restype = ci
    lib.siren_b200_comm_init.argtypes = [ci, ci, vp, ctypes.POINTER(ctypes.c_void_p)]
    lib.siren_b200_allreduce.restype = ci
    lib.siren_b200_allreduce.argtypes = [vp, fp, cl, vp]
    lib.siren_b200_allreduce_peers.restype = ci
    lib.siren_b200_allreduce_peers.argtypes = [vp, ci, ci, cl, cf, vp]
    lib.siren_b200_allreduce_multicast.restype = ci
    lib.siren_b200_allreduce_multicast.argtypes = [vp, ci, ci, cl, cf, vp]
    lib.siren_b200_comm_destroy.restype = ci
    lib.siren_b200_comm_destroy.argtypes = [vp]
    lib.siren_b200_comm_last_error.restype = ctypes.c_char_p
    lib.siren_b200_debug_linear.restype = ci
    lib.siren_b200_debug_linear.argtypes = [fp, fp, fp, cl, ci, vp, vp]
    lib.siren_b200_debug_wgrad.restype = ci
    lib.siren_b200_debug_wgrad.argtypes = [fp, fp, fp, cl, ci, vp, vp]
    return lib


def load():
    """Return the bound library, loading it on first use.  Raises NativeError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(
                    "siren_mri_b200: native library not built (%s missing). Run "
                    "`make -C siren_mri_b200/csrc -j` or `python -c 'import __graft_entry__ as g; g.build()'`."
                    % LIB_PATH)
            try:
                lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
            except OSError as e:  # pragma: no cover
                raise NativeError("siren_mri_b200: cannot load %s: %s" % (LIB_PATH, e)) from e
            _lib = _bind(lib)
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().siren_b200_last_error()
        raise NativeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr_array(tensors):
    """Host array of device pointers for a list of tensors (None -> NULL)."""
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def ptr_array_raw(addresses):
    """Host array of device pointers from raw addresses."""
    arr = (ctypes.c_void_p * len(addresses))()
    for i, a in enumerate(addresses):
        arr[i] = a
    return arr


def dptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())
