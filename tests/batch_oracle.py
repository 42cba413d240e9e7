"""CPU oracle of the greedy batch acquisition (MultifidelityDataFusion.acquisition_batch), by its definition: q
sequential candidate-set acquisitions at FIXED hyper-parameters, each refactorising the augmented training set plus
the picks so far with GPy's arithmetic (oracle/gpy_oracle.py: K + (noise + 1e-8) I, jitchol, 1e-15 clip, + noise).
Kept beside the tests that use it; oracle/ holds the restatement of the reference and stays as it is."""
import numpy as np

from oracle import gpy_oracle as go


def candidate_batch(model, candidates, q):
    """model: a fitted oracle.mfgp_oracle.OracleMFGP.  Returns (indices (q,), variances (q,) with noise,
    top-2 relative gaps (q,)).  The targets of the picks never enter: the predictive variance does not depend on
    them, so zeros stand in for f_exact."""
    hf = model.hf_model
    theta = hf.theta.copy()
    if model.add_noise:                                             # MFDataFusion.py:154-155
        theta[-1] = 1e-6
    Xc = model.augment(np.ascontiguousarray(candidates, dtype=np.float64))
    X = hf.X.copy()
    idx, var, gaps = [], [], []
    for _ in range(int(q)):
        g = go.OracleGPRegression(X, np.zeros((X.shape[0], 1)), hf.kind, d=hf.d, theta=theta, form=hf.form)
        v = g.predict(Xc)[1].ravel()
        i = int(np.argmax(v))
        second = np.partition(v, -2)[-2] if v.size > 1 else -np.inf
        idx.append(i)
        var.append(float(v[i]))
        gaps.append(float((v[i] - second) / abs(v[i])) if v[i] != 0 else 0.0)
        X = np.vstack([X, Xc[i]])
    return np.array(idx, dtype=np.int64), np.array(var), np.array(gaps)
