"""Tensor-level wrappers of the C-ABI calls (torch CUDA float64 tensors in, tensors out).

Thin by design: argument marshalling only.  Used by the parity tests and bench.py to drive single
kernels; the model classes go through ``gp.GPRegression``.
"""
import ctypes

import numpy as np
import torch

from . import _ffi
from ._ffi import KIND_COMPOSITE, KIND_RBF, UPLO_FULL, UPLO_LOWER, padded_n


def _theta(theta):
    arr = (ctypes.c_double * 8)()
    for i, v in enumerate(np.asarray(theta, dtype=np.float64).ravel()):
        arr[i] = float(v)
    return arr, len(np.asarray(theta).ravel())


def _dev(t):
    assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
    return t.device.index


def assemble(X, kind, d, theta, uplo=UPLO_LOWER, jitter=0.0, ld=None):
    """K1.  X (N,D) -> K_y (N, ld) with K + (noise + 1e-8 + jitter) I in [:, :N]."""
    dev = _dev(X)
    h = _ffi.get_handle(dev)
    N, D = X.shape
    ld = N if ld is None else ld
    K = torch.zeros((N, ld), dtype=torch.float64, device=X.device)
    th, P = _theta(theta)
    h.check(h.lib.mfgp_assemble(h.h, kind, X.data_ptr(), N, D, d, ctypes.cast(th, ctypes.c_void_p), P,
                                float(jitter), K.data_ptr(), ld, uplo))
    return K


def pad_spd(A):
    """Embed an (n,n) SPD matrix in the (npad,npad) identity-padded layout the factor kernels use."""
    n = A.shape[0]
    npad = padded_n(n)
    P = torch.eye(npad, dtype=torch.float64, device=A.device)
    P[:n, :n] = A
    return P


def potrf(Apad):
    """In place: Apad (npad,npad) -> L (lower).  Returns (W with the 128-leaf inverses, info)."""
    h = _ffi.get_handle(_dev(Apad))
    npad = Apad.shape[0]
    W = torch.zeros_like(Apad)
    info = h.lib.mfgp_potrf(h.h, Apad.data_ptr(), W.data_ptr(), npad)
    if info < 0:
        h.check(info)
    return W, info


def trtri(Lpad, W):
    h = _ffi.get_handle(_dev(Lpad))
    h.check(h.lib.mfgp_trtri(h.h, Lpad.data_ptr(), W.data_ptr(), Lpad.shape[0]))
    return W


def lauum(W):
    h = _ffi.get_handle(_dev(W))
    Kinv = torch.zeros_like(W)
    h.check(h.lib.mfgp_lauum(h.h, W.data_ptr(), Kinv.data_ptr(), W.shape[0]))
    return Kinv


class FactorBuffers:
    """Caller-owned buffers of one GP level: A (K_y -> L -> K^-1), W (L^-1), alpha."""

    def __init__(self, N, device):
        self.N, self.npad = N, padded_n(N)
        self.A = torch.empty((self.npad, self.npad), dtype=torch.float64, device=device)
        self.W = torch.empty((self.npad, self.npad), dtype=torch.float64, device=device)
        self.alpha = torch.empty(self.npad, dtype=torch.float64, device=device)


def factorize(X, y, kind, d, theta, buf, jitter=0.0):
    """K1-K3.  Returns (lml, logdet, yTalpha, info); buf.A = L, buf.W = L^-1, buf.alpha."""
    h = _ffi.get_handle(_dev(X))
    N, D = X.shape
    th, P = _theta(theta)
    out = (ctypes.c_double * 3)()
    info = h.lib.mfgp_factorize(h.h, kind, X.data_ptr(), y.data_ptr(), N, D, d,
                                ctypes.cast(th, ctypes.c_void_p), P, float(jitter), buf.A.data_ptr(),
                                buf.W.data_ptr(), buf.alpha.data_ptr(), ctypes.cast(out, ctypes.c_void_p))
    if info < 0:
        h.check(info)
    return out[0], out[1], out[2], info


def lml_grad(X, y, kind, d, theta, buf, jitter=0.0, timed=False):
    """K1-K5.  Returns (lml, grad (P,), info[, stage_ms (6,)]); buf.A = K^-1 (lower)."""
    h = _ffi.get_handle(_dev(X))
    N, D = X.shape
    th, P = _theta(theta)
    lml = ctypes.c_double()
    grad = (ctypes.c_double * 8)()
    ms = (ctypes.c_double * 8)()
    info = h.lib.mfgp_lml_grad_timed(h.h, kind, X.data_ptr(), y.data_ptr(), N, D, d,
                                     ctypes.cast(th, ctypes.c_void_p), P, float(jitter),
                                     buf.A.data_ptr(), buf.W.data_ptr(), buf.alpha.data_ptr(),
                                     ctypes.byref(lml), ctypes.cast(grad, ctypes.c_void_p),
                                     ctypes.cast(ms, ctypes.c_void_p) if timed else None)
    if info < 0:
        h.check(info)
    g = np.array([grad[i] for i in range(P)])
    if timed:
        return lml.value, g, info, np.array([ms[i] for i in range(6)])
    return lml.value, g, info


class LevelRef:
    """Keeps an mfgp_level_t and the buffers it points to alive."""

    def __init__(self, X, kind, d, theta, buf):
        self.X, self.buf = X, buf
        self.theta, P = _theta(theta)
        self.struct = _ffi.Level(kind=kind, N=X.shape[0], D=X.shape[1], d=d, P=P, reserved=0,
                                 d_X=X.data_ptr(), h_theta=ctypes.cast(self.theta, ctypes.c_void_p).value,
                                 d_W=buf.W.data_ptr(), d_alpha=buf.alpha.data_ptr())

    @property
    def ref(self):
        return ctypes.byref(self.struct)


def predict(level, Xnew, want_var=True, include_noise=True, ws_bytes=None):
    h = _ffi.get_handle(_dev(Xnew))
    M = Xnew.shape[0]
    mean = torch.empty(M, dtype=torch.float64, device=Xnew.device)
    var = torch.empty(M, dtype=torch.float64, device=Xnew.device) if want_var else None
    N = level.struct.N
    if ws_bytes is None:
        ws_bytes = min(max(h.lib.mfgp_predict_ws_bytes(N, max(M, 1)), 1), 1 << 30)
        ws_bytes = max(ws_bytes, h.lib.mfgp_predict_ws_bytes(N, 128))
    ws = torch.empty((ws_bytes + 7) // 8, dtype=torch.float64, device=Xnew.device)
    h.check(h.lib.mfgp_predict(h.h, level.ref, Xnew.data_ptr(), M, mean.data_ptr(),
                               var.data_ptr() if want_var else None, int(include_noise),
                               ws.data_ptr(), ws.numel() * 8))
    return mean, var


def predictive_gradients(level, Xnew, want_var=True, include_noise=True, ws_bytes=None):
    """K6d.  Xnew (M, D) -> (dmean (M, D), dvar (M, D) or None, mean (M,), var (M,) or None); dvar is the gradient
    of the unclipped latent variance, mean and var are predict's outputs to round-off.  want_var=False: mean-only
    mode (no W, no scratch)."""
    h = _ffi.get_handle(_dev(Xnew))
    M, D = Xnew.shape
    if D != level.struct.D:
        raise ValueError("Xnew has %d columns, the level has D = %d" % (D, level.struct.D))
    new = lambda *shape: torch.empty(shape, dtype=torch.float64, device=Xnew.device)
    dmean, mean = new(M, D), new(M)
    dvar, var, ws, nbytes = None, None, None, 0
    if want_var:
        dvar, var = new(M, D), new(M)
        N = level.struct.N
        if ws_bytes is None:
            ws_bytes = max(min(h.lib.mfgp_predictive_gradients_ws_bytes(N, max(M, 1)), 1 << 30),
                           h.lib.mfgp_predictive_gradients_ws_bytes(N, 128))
        ws = new((ws_bytes + 7) // 8)
        nbytes = ws.numel() * 8
    ptr = lambda t: t.data_ptr() if t is not None else None
    h.check(h.lib.mfgp_predictive_gradients(h.h, level.ref, Xnew.data_ptr(), M, dmean.data_ptr(), ptr(dvar),
                                            mean.data_ptr(), ptr(var), int(include_noise), ptr(ws), nbytes))
    return dmean, dvar, mean, var


def fill_normal(seed, first, count, device):
    h = _ffi.get_handle(torch.device(device).index or 0)
    out = torch.empty(count, dtype=torch.float64, device=device)
    h.check(h.lib.mfgp_fill_normal(h.h, int(seed), int(first), int(count), out.data_ptr()))
    return out


def argmax(v):
    h = _ffi.get_handle(_dev(v))
    val, idx = ctypes.c_double(), ctypes.c_longlong()
    h.check(h.lib.mfgp_argmax(h.h, v.data_ptr(), v.numel(), ctypes.byref(val), ctypes.byref(idx)))
    return val.value, idx.value
