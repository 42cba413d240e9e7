"""Predictive gradients of a GP level and of the multi-fidelity chain rule, restated in NumPy on the oracle's kernel
parts (GPy's ``GP.predictive_gradients``): an independent formulation for the tests of mfgp_predictive_gradients.

    dmean[c][j] = sum_k alpha_k dk(q_c, X_k)/dq_j,   dvar[c][j] = -2 sum_k u_kc dk(q_c, X_k)/dq_j,  u = K_y^-1 k

dvar is the gradient of the unclipped latent variance (k(q, q) is constant)."""
import numpy as np
from scipy.linalg import cho_solve

from oracle import gpy_oracle as go


def kernel_grad(kind, X, Xq, d, theta_k):
    """(M, N, D): dk(q_c, X_k) / dq_j from kernel_K's parts (RBF: s exp(-r^2/2), r = |q - x| / l)."""
    _, parts = go.kernel_K(kind, Xq, X, d, theta_k, form="direct", want_parts=True)
    diff = Xq[:, None, :] - X[None, :, :]                                 # (M, N, D)
    if kind == go.KIND_RBF:
        return -diff * (parts["K1"] / theta_k[1] ** 2)[:, :, None]
    K12 = parts["K1"] * parts["K2"]
    g = np.empty_like(diff)
    g[:, :, :d] = -diff[:, :, :d] * (K12 / theta_k[3] ** 2 + parts["K3"] / theta_k[5] ** 2)[:, :, None]
    g[:, :, d:] = -diff[:, :, d:] * (K12 / theta_k[1] ** 2)[:, :, None]
    return g


def level_gradients(kind, X, Y, d, theta, Xq):
    """(dmean (M, D), dvar (M, D)) of the level fitted on (X, Y) at fixed theta."""
    res = go.inference(kind, X, Y, d, theta, form="direct", want_grad=False)
    theta_k, _ = go.split_theta(kind, theta)
    dK = kernel_grad(kind, X, Xq, d, theta_k)
    Kx = go.kernel_K(kind, X, Xq, d, theta_k, form="direct")              # (N, M)
    u = cho_solve((res["L"], True), Kx)
    dmean = np.einsum("mnj,n->mj", dK, res["alpha"].ravel())
    dvar = -2.0 * np.einsum("mnj,nm->mj", dK, u)
    return dmean, dvar


def mf_gradients(hf_grads, X, offsets, tau, f_low_jac):
    """Chain rule through x -> [x, f_low(x + o_e tau)]: hf_grads(Xa) -> (dmean, dvar) on augmented rows, f_low_jac
    (n, d) locations -> (n, d).  Returns (dmean (M, d), dvar (M, d)) with respect to x."""
    M, d = X.shape
    E = offsets.shape[0]
    gm, gv = hf_grads
    J = f_low_jac((X[:, None, :] + offsets[None, :, :] * tau).reshape(M * E, d)).reshape(M, E, d)
    return (gm[:, :d] + np.einsum("me,med->md", gm[:, d:], J),
            gv[:, :d] + np.einsum("me,med->md", gv[:, d:], J))


def central_diff(fun, X, h=1e-6):
    """(M, d) derivative of a row-wise fun (M, d) -> (M,) by central differences."""
    X = np.asarray(X, dtype=np.float64)
    out = np.empty_like(X)
    for j in range(X.shape[1]):
        e = np.zeros(X.shape[1])
        e[j] = h
        out[:, j] = (fun(X + e) - fun(X - e)) / (2 * h)
    return out
