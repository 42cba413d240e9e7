"""Predictive gradients and the multi-start L-BFGS-B acquisition on the GPU.

(a) mfgp_predictive_gradients against mfgp_predict on the same batch: a composite level with N_h = 1024 (D = 5, the
    high-fidelity level of bench.py's acquisition model, whose data-driven LF level has N_l = 4096) and M = 2^16
    queries; CUDA events around each call after a warm-up, median of --reps; plus the multi-fidelity call
    (MultifidelityDataFusion.predictive_gradients_device: augmentation, HF gradients, LF mean-only gradients, chain
    rule) at the same M.
(b) one acquisition at the config-2 (GPDF 2-D, 10^5 candidates) and config-3 (NARGP 4-D, 2^20 candidates) shapes with
    DIRECT through the resident point service (ScipyDirectMaximizer), CandidateSetMaximizer and LBFGSBMaximizer:
    wall time between device synchronisations (after one warm-up acquisition), the variance predict reports at the
    returned point, and the L-BFGS-B rounds (batched gradient calls).
Records the card's name and power limit in the same run.  Writes DIR/acq_lbfgsb_probe.json.

    python tools/acq_lbfgsb_probe.py --out DIR [--reps 5]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from acq_batch_probe import card, hf_4d, lf_4d, shapes  # noqa: E402


def events_ms(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def part_a(pkg, gp, reps):
    rng = np.random.default_rng(1)
    Xh, Xl = rng.uniform(size=(1024, 4)), rng.uniform(size=(4096, 4))
    m = pkg.NARGP(4, hf_4d, None, lf_X=Xl, lf_Y=hf_4d(Xl) - 0.1)
    m.lf_model._set_params(np.array([1.0, 0.3, 1e-3]))
    m.fit(Xh, theta=np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 1e-3]))
    M = 1 << 16
    dX = gp.to_device(rng.uniform(size=(M, 4)), m.device)
    dXa = m._augment_device(dX)
    hf = m.hf_model
    t_pred = events_ms(lambda: hf.predict_device(dXa, True, True), reps)
    t_grad = events_ms(lambda: hf.predictive_gradients_device(dXa, True, True), reps)
    t_mean = events_ms(lambda: hf.predictive_gradients_device(dXa, False), reps)
    t_mf = events_ms(lambda: m.predictive_gradients_device(dX), reps)
    _, _, mean, var = hf.predictive_gradients_device(dXa, True, True)
    pm, pv = hf.predict_device(dXa, True, True)
    return {"N_h": hf.N, "N_l": m.lf_model.N, "D": hf.D, "M": M,
            "predict_ms": float(np.median(t_pred)), "predict_ms_all": t_pred,
            "predictive_gradients_ms": float(np.median(t_grad)), "predictive_gradients_ms_all": t_grad,
            "ratio_to_predict": float(np.median(t_grad) / np.median(t_pred)),
            "mean_only_gradients_ms": float(np.median(t_mean)),
            "mf_predictive_gradients_ms": float(np.median(t_mf)), "mf_predictive_gradients_ms_all": t_mf,
            "max_abs_mean_vs_predict": float((mean - pm).abs().max()),
            "max_abs_var_vs_predict": float((var - pv).abs().max())}


def part_b(pkg, gp, reps):
    import torch
    out = {}
    for name, (factory, cands) in shapes(pkg, gp).items():
        if name.startswith("bench"):
            continue
        rows = {}
        for label, make in (("direct", lambda: pkg.ScipyDirectMaximizer()),
                            ("candidate_set", lambda: pkg.CandidateSetMaximizer(candidates=cands)),
                            ("lbfgsb", lambda: pkg.LBFGSBMaximizer(candidates=cands))):
            m = factory()
            lb, ub = np.zeros(m.input_dim), np.ones(m.input_dim)
            make().maximize(m.predict, lb, ub)              # warm-up: candidates resident, kernels paged in
            ts = []
            for _ in range(1 if label == "direct" else reps):
                mx = make()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                x, fopt = mx.maximize(m.predict, lb, ub)
                torch.cuda.synchronize()
                ts.append(1e3 * (time.perf_counter() - t0))
            rows[label] = {"ms": float(np.median(ts)), "ms_all": ts, "variance": -float(fopt),
                           "x": [float(v) for v in x], "rounds": getattr(mx, "last_rounds", None)}
            print(name, label, "%.1f ms" % rows[label]["ms"], "variance %.6e" % rows[label]["variance"], flush=True)
        out[name] = {"candidates": int(cands.shape[0]), "N_h": 30, "by_maximizer": rows}
        gp.release_workspaces()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import multifidelity_datafusion_gps_b200 as pkg
    from multifidelity_datafusion_gps_b200 import gp
    os.makedirs(args.out, exist_ok=True)
    res = {"card": card(), "reps": args.reps}
    res["gradients_vs_predict"] = part_a(pkg, gp, args.reps)
    print(json.dumps(res["gradients_vs_predict"]), flush=True)
    res["acquisition"] = part_b(pkg, gp, args.reps)
    with open(os.path.join(args.out, "acq_lbfgsb_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
