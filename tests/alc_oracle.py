"""CPU oracle of the integrated-variance (ALC) acquisition (GPRegression.alc_device, mfgp_alc), on augmented rows and
with GPy's arithmetic (oracle/gpy_oracle.py: K + (noise + 1e-8) I, jitchol).  Two independent formulations:
  closed_form  alc(c) = sum_r w_r k_n(c, r)^2 / (v_n(c) + s^2),  s^2 = noise + 1e-8 + jitter
  definition   alc(c) = sum_r w_r (v_n(r) - v_{n+c}(r)), refactorising X + {c} at the same theta
Kept beside the tests that use it; oracle/ holds the restatement of the reference and stays as it is."""
import numpy as np
from scipy.linalg import solve_triangular

from oracle import gpy_oracle as go


def _factor(kind, X, d, theta, form):
    """(L, jitter) of K_y + jitter I as jitchol leaves it."""
    return go.jitchol(go.assemble_Ky(kind, X, d, theta, form))


def _weights(w, R):
    return np.full(R, 1.0 / R) if w is None else np.asarray(w, dtype=np.float64)


def closed_form(kind, X, d, theta, Xc, Xr, w=None, form="direct", chunk=4096):
    """(C,) ALC values from the latent posterior covariance; -inf where v_n(c) + s^2 <= 0.  Candidates are scored
    in chunks so that C x R blocks stay small."""
    theta_k, noise = go.split_theta(kind, theta)
    L, jitter = _factor(kind, X, d, theta, form)
    s2 = noise + go.JITTER_CONST + jitter
    w = _weights(w, Xr.shape[0])
    Tr = solve_triangular(L, go.kernel_K(kind, X, Xr, d, theta_k, form), lower=True)          # (N, R)
    kdiag = go.kernel_Kdiag(kind, theta_k, 1)[0]
    out = np.empty(Xc.shape[0])
    for c0 in range(0, Xc.shape[0], chunk):
        xc = Xc[c0:c0 + chunk]
        Tc = solve_triangular(L, go.kernel_K(kind, X, xc, d, theta_k, form), lower=True)      # (N, c)
        kn = go.kernel_K(kind, xc, Xr, d, theta_k, form) - Tc.T @ Tr                          # (c, R)
        den = kdiag - np.sum(Tc * Tc, axis=0) + s2
        with np.errstate(divide="ignore", invalid="ignore"):
            out[c0:c0 + chunk] = np.where(den > 0.0, (kn * kn) @ w / den, -np.inf)
    return out


def latent_variance(kind, X, d, theta, Xr, jitter_extra=None, form="direct"):
    """Unclipped latent variance at Xr of the GP on X; jitter_extra (the jitter of the factor being extended) is
    added to the diagonal instead of running jitchol's schedule when given."""
    theta_k, _ = go.split_theta(kind, theta)
    Ky = go.assemble_Ky(kind, X, d, theta, form)
    if jitter_extra is None:
        L, _ = go.jitchol(Ky)
    else:
        L = np.linalg.cholesky(Ky + jitter_extra * np.eye(Ky.shape[0]))
    T = solve_triangular(L, go.kernel_K(kind, X, Xr, d, theta_k, form), lower=True)
    return go.kernel_Kdiag(kind, theta_k, Xr.shape[0]) - np.sum(T * T, axis=0)


def definition(kind, X, d, theta, Xc, Xr, w=None, form="direct"):
    """(C,) ALC values by refactorising X + {c} at fixed theta (and the jitter of the N-point factor, as
    append_point keeps it) and summing the weighted variance drop at the references."""
    _, jitter = _factor(kind, X, d, theta, form)
    w = _weights(w, Xr.shape[0])
    before = latent_variance(kind, X, d, theta, Xr, jitter, form)
    return np.array([w @ (before - latent_variance(kind, np.vstack([X, c]), d, theta, Xr, jitter, form))
                     for c in Xc])


def sequential_picks(kind, X, d, theta, Xc, Xr, steps, w=None, form="direct"):
    """What `steps` ALC adaptation steps at fixed theta pick: refactorise, rescore, append the winner, repeat.
    Returns (indices, alc values, top-2 relative gaps)."""
    idx, vals, gaps = [], [], []
    for _ in range(int(steps)):
        a = closed_form(kind, X, d, theta, Xc, Xr, w, form)
        i = int(np.argmax(a))
        second = np.partition(a, -2)[-2] if a.size > 1 else -np.inf
        idx.append(i)
        vals.append(float(a[i]))
        gaps.append(float((a[i] - second) / abs(a[i])) if a[i] != 0 else 0.0)
        X = np.vstack([X, Xc[i]])
    return np.array(idx, dtype=np.int64), np.array(vals), np.array(gaps)
