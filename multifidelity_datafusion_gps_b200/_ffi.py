"""ctypes binding of include/mfgp_b200.h (the C-ABI boundary).

PyTorch is only the tensor carrier: every pointer handed to the library is the ``data_ptr()``
of a contiguous float64 / int64 CUDA tensor.  There is NO fallback: if the shared library is
missing, or no B200 is present, the first call raises.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# MFGP_LIB: kernel-tuning override (tools/build_variants.sh builds A/B variants of the same library)
LIB_PATH = os.environ.get("MFGP_LIB") or os.path.join(_HERE, "libmfgp_b200.so")

KIND_RBF = 0
KIND_COMPOSITE = 1
UPLO_LOWER = 0
UPLO_FULL = 1
TILE = 128
ACQ_MAX_Q = 64           # MFGP_ACQ_MAX_Q: largest batch of mfgp_acq_batch_*

EXPORTS = [
    "mfgp_version", "mfgp_padded_n", "mfgp_create", "mfgp_destroy", "mfgp_set_stream",
    "mfgp_last_error", "mfgp_launch_count", "mfgp_profile_enable", "mfgp_profile_read", "mfgp_assemble", "mfgp_factorize", "mfgp_lml_grad",
    "mfgp_lml_grad_timed", "mfgp_lml_grad_batch_max", "mfgp_lml_grad_batch", "mfgp_append_point", "mfgp_potrf", "mfgp_trtri", "mfgp_lauum", "mfgp_predict_ws_bytes",
    "mfgp_predict", "mfgp_predict_small_max_rows", "mfgp_predict_small", "mfgp_point_service_start", "mfgp_point_service_eval", "mfgp_point_service_stop", "mfgp_point_service_relaunches", "mfgp_augment", "mfgp_predict_mc_ws_bytes", "mfgp_predict_mc", "mfgp_predict_mc_chain", "mfgp_predict_mc_joint_ws_bytes", "mfgp_predict_mc_joint",
    "mfgp_predict_mc_delays", "mfgp_fill_normal",
    "mfgp_predictive_gradients_ws_bytes", "mfgp_predictive_gradients",
    "mfgp_argmax", "mfgp_acq_batch_ws_bytes", "mfgp_acq_batch_begin", "mfgp_acq_batch_step",
    "mfgp_alc_ws_bytes", "mfgp_alc",
    "mfgp_pce_ws_bytes", "mfgp_pce_project",
]


class MfgpError(RuntimeError):
    pass


class NotPositiveDefinite(MfgpError):
    """LAPACK-style info > 0 from the Cholesky factorisation (first bad pivot, 1-based)."""

    def __init__(self, info):
        super().__init__("covariance not positive definite (first bad pivot %d)" % info)
        self.info = info


class Level(ctypes.Structure):
    """mfgp_level_t"""
    _fields_ = [("kind", ctypes.c_int32), ("N", ctypes.c_int32), ("D", ctypes.c_int32),
                ("d", ctypes.c_int32), ("P", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("d_X", ctypes.c_void_p), ("h_theta", ctypes.c_void_p),
                ("d_W", ctypes.c_void_p), ("d_alpha", ctypes.c_void_p)]


_lib = None


def load_library():
    """Load libmfgp_b200.so and declare every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MfgpError(
            "libmfgp_b200.so is not built (%s). Run `python __graft_entry__.py` or "
            "`python multifidelity_datafusion_gps_b200/build.py`; there is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    c_int, c_ll, c_dbl, vp = ctypes.c_int, ctypes.c_longlong, ctypes.c_double, ctypes.c_void_p
    c_ull, c_sz = ctypes.c_ulonglong, ctypes.c_size_t
    lib.mfgp_version.restype = c_int
    lib.mfgp_padded_n.argtypes = [c_int]
    lib.mfgp_create.argtypes = [c_int, ctypes.POINTER(vp)]
    lib.mfgp_destroy.argtypes = [vp]
    lib.mfgp_set_stream.argtypes = [vp, vp]
    lib.mfgp_last_error.argtypes = [vp]
    lib.mfgp_last_error.restype = ctypes.c_char_p
    lib.mfgp_launch_count.argtypes = [vp]
    lib.mfgp_launch_count.restype = c_ll
    lib.mfgp_profile_enable.argtypes = [vp, c_int]
    lib.mfgp_profile_read.argtypes = [vp, vp, vp]
    lib.mfgp_assemble.argtypes = [vp, c_int, vp, c_int, c_int, c_int, vp, c_int, c_dbl, vp, c_ll, c_int]
    lib.mfgp_factorize.argtypes = [vp, c_int, vp, vp, c_int, c_int, c_int, vp, c_int, c_dbl, vp, vp, vp, vp]
    lib.mfgp_append_point.argtypes = [vp, c_int, vp, vp, c_int, c_int, c_int, vp, c_int, c_dbl, vp, vp, vp, c_int, vp]
    lib.mfgp_lml_grad.argtypes = [vp, c_int, vp, vp, c_int, c_int, c_int, vp, c_int, c_dbl, vp, vp, vp, vp, vp]
    lib.mfgp_lml_grad_timed.argtypes = lib.mfgp_lml_grad.argtypes + [vp]
    lib.mfgp_lml_grad_batch.argtypes = [vp, c_int, vp, vp, c_int, c_int, c_int, vp, c_int, c_int, c_dbl, vp, vp, vp]
    lib.mfgp_potrf.argtypes = [vp, vp, vp, c_int]
    lib.mfgp_trtri.argtypes = [vp, vp, vp, c_int]
    lib.mfgp_lauum.argtypes = [vp, vp, vp, c_int]
    lib.mfgp_predict_ws_bytes.argtypes = [c_int, c_ll]
    lib.mfgp_predict_ws_bytes.restype = c_sz
    lib.mfgp_predict.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, vp, vp, c_int, vp, c_sz]
    lib.mfgp_predict_small.argtypes = [vp, ctypes.POINTER(Level), ctypes.POINTER(Level), vp, c_int, vp, c_int,
                                       c_dbl, c_int, vp, vp]
    lib.mfgp_augment.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, vp, c_int, c_dbl, vp, vp, c_sz]
    lib.mfgp_predict_mc.argtypes = [vp, ctypes.POINTER(Level), ctypes.POINTER(Level), vp, c_ll, c_int,
                                    vp, c_ull, c_ll, c_int, c_int, vp, vp, vp, vp, vp, c_sz]
    lib.mfgp_predict_mc_chain.argtypes = [vp, vp, c_int, vp, c_ll, c_int, vp, c_ull, c_ll, c_int, c_int, vp, vp,
                                          vp, vp, vp, c_sz]
    lib.mfgp_point_service_start.argtypes = [vp, ctypes.POINTER(Level), ctypes.POINTER(Level), vp, c_int, c_dbl, c_int,
                                             c_dbl]
    lib.mfgp_point_service_eval.argtypes = [vp, vp, vp]
    lib.mfgp_point_service_stop.argtypes = [vp]
    lib.mfgp_point_service_relaunches.argtypes = [vp]
    lib.mfgp_point_service_relaunches.restype = c_ll
    lib.mfgp_predict_mc_ws_bytes.argtypes = [c_int, c_int, c_int, c_ll, c_int]
    lib.mfgp_predict_mc_ws_bytes.restype = c_sz
    lib.mfgp_predict_mc_joint_ws_bytes.argtypes = [c_int, c_int, c_ll, c_int]
    lib.mfgp_predict_mc_joint_ws_bytes.restype = c_sz
    lib.mfgp_predict_mc_joint.argtypes = [vp, ctypes.POINTER(Level), ctypes.POINTER(Level), vp, c_ll, c_int, vp,
                                          c_ull, c_int, c_int, c_dbl, vp, vp, vp, vp, vp, c_sz]
    lib.mfgp_predict_mc_delays.argtypes = [vp, ctypes.POINTER(Level), ctypes.POINTER(Level), vp, c_ll, vp, c_int,
                                           c_dbl, c_int, vp, c_ull, c_ll, c_int, c_int, c_dbl, vp, vp, vp, vp,
                                           vp, c_sz]
    lib.mfgp_fill_normal.argtypes = [vp, c_ull, c_ll, c_ll, vp]
    lib.mfgp_argmax.argtypes = [vp, vp, c_ll, vp, vp]
    lib.mfgp_predictive_gradients_ws_bytes.argtypes = [c_int, c_ll]
    lib.mfgp_predictive_gradients_ws_bytes.restype = c_sz
    lib.mfgp_predictive_gradients.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, vp, vp, vp, vp, c_int, vp, c_sz]
    lib.mfgp_alc_ws_bytes.argtypes = [c_int, c_ll, c_ll]
    lib.mfgp_alc_ws_bytes.restype = c_sz
    lib.mfgp_alc.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, vp, c_ll, vp, c_dbl, vp, vp, c_sz]
    lib.mfgp_acq_batch_ws_bytes.argtypes = [c_int, c_ll, c_int]
    lib.mfgp_acq_batch_ws_bytes.restype = c_sz
    lib.mfgp_acq_batch_begin.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, c_int, c_int, vp, c_sz, vp, vp, vp]
    lib.mfgp_acq_batch_step.argtypes = [vp, ctypes.POINTER(Level), vp, c_ll, c_int, c_int, c_dbl, c_int, vp, vp, c_sz,
                                        vp, vp, vp]
    lib.mfgp_pce_ws_bytes.argtypes = [c_int, c_int]
    lib.mfgp_pce_ws_bytes.restype = c_sz
    lib.mfgp_pce_project.argtypes = [vp, vp, vp, vp, c_int, vp, vp, c_ll, vp, c_int, c_int, vp, vp, vp, c_sz]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("mfgp_last_error", "mfgp_launch_count", "mfgp_predict_ws_bytes", "mfgp_pce_ws_bytes",
                        "mfgp_predict_mc_joint_ws_bytes", "mfgp_predict_mc_ws_bytes", "mfgp_point_service_relaunches",
                        "mfgp_acq_batch_ws_bytes", "mfgp_predictive_gradients_ws_bytes", "mfgp_alc_ws_bytes"):
            fn.restype = c_int
    _lib = lib
    return lib


def padded_n(n):
    return (max(int(n), 1) + TILE - 1) // TILE * TILE


class Handle:
    """Owns one mfgp_handle_t (one per GPU / per Python thread)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.mfgp_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise MfgpError("mfgp_create failed (%d): %s" %
                            (rc, self.lib.mfgp_last_error(None).decode()))
        self.h = h
        self.device = int(device)
        self._stream_ptr = None                 # stream the C side is bound to (get_handle keeps it current)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mfgp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        """0 -> ok; >0 -> NotPositiveDefinite; <0 -> MfgpError with the library's message."""
        if rc == 0:
            return
        if rc > 0:
            raise NotPositiveDefinite(rc)
        raise MfgpError("mfgp call failed (%d): %s" % (rc, self.lib.mfgp_last_error(self.h).decode()))

    def set_stream(self, stream_ptr):
        self.check(self.lib.mfgp_set_stream(self.h, ctypes.c_void_p(stream_ptr)))

    PROFILE_CLASSES = ["assemble", "potrf_leaf", "gemm", "solve", "lauum", "grad_reduce", "cross_gen",
                       "trmm_sumsq", "misc", "argmax"]

    def profile_enable(self, on=True):
        self.check(self.lib.mfgp_profile_enable(self.h, int(on)))

    def profile_read(self):
        """{class: (average launch ms, launches)} since profile_enable."""
        ms = (ctypes.c_double * 16)()
        cnt = (ctypes.c_longlong * 16)()
        self.check(self.lib.mfgp_profile_read(self.h, ctypes.cast(ms, ctypes.c_void_p),
                                              ctypes.cast(cnt, ctypes.c_void_p)))
        return {n: (ms[i], int(cnt[i])) for i, n in enumerate(self.PROFILE_CLASSES)}

    @property
    def launches(self):
        return int(self.lib.mfgp_launch_count(self.h))


_handles = {}
_handles_lock = threading.Lock()


def get_handle(device=0):
    """One handle per (device, Python thread), bound to torch's current stream on that device.
    A handle owns its stream binding, result staging and scratch, and ctypes releases the GIL during
    calls, so two threads must never share one (include/mfgp_b200.h: thread-compatible per handle)."""
    import torch
    if not torch.cuda.is_available():
        raise MfgpError("no CUDA device visible: mfgp_b200 has no CPU fallback")
    key = (int(device), threading.get_ident())
    h = _handles.get(key)
    if h is None:
        with _handles_lock:
            h = _handles[key] = Handle(int(device))
    sp = torch.cuda.current_stream(int(device)).cuda_stream
    if sp != h._stream_ptr:                     # (re)bind only when torch's current stream changed
        h.set_stream(sp)
        h._stream_ptr = sp
    return h


def total_launches(device=None):
    """Kernels launched by every handle of this process (optionally of one device)."""
    return sum(h.launches for (dev, _), h in list(_handles.items()) if device is None or dev == int(device))
