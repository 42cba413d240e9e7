"""Integrated-variance (ALC) acquisition against the variance arg-max, on the GPU.

For the three shapes of bench.py's acquisition block (tools/acq_batch_probe.py: config 2, config 3 and the N_h = 1024
bench model) and R in {256, 1024, 4096} reference rows: wall time of a resident acquisition_alc against
acquisition_argmax on the same candidates, each timed region between device synchronisations after a warm-up; the
per-class kernel times of one ALC call (mfgp_profile_*: 6 the K(., X) blocks, 8 the Tt = Ks W^T products, 2 the
G = Tt_C Tt_R^T product, 9 the fused ALC reduction); the flops the products need (C Npad^2 + 2 C R Npad + R Npad^2)
and the bytes of G (16 C R, written once and read once): the flops as a rate against the cuBLAS DGEMM 8192^3 rate
measured in the same run, the bytes as the time they take at the data sheet's 7.7 TB/s (a floor, not a measurement); and the card's name and power limit.  For information only: the test MSE after 10 adaptation steps of
config 2 with CandidateSetMaximizer and with ALCMaximizer on the same candidates.  Writes DIR/acq_alc_probe.json.

    python tools/acq_alc_probe.py --out DIR [--reps 3]
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

from acq_batch_probe import card, hf_2d, lf_2d, shapes  # noqa: E402

CLASS_NAMES = {"cross_gen": "K(., X) blocks", "misc": "Tt = Ks W^T", "gemm": "G = Tt_C Tt_R^T",
               "argmax": "ALC reduction + arg-max"}


def dgemm_rate(torch):
    """cuBLAS DGEMM 8192^3 in TFLOP/s, best of five after a warm-up (bench.py's measuring stick)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    best = 1e30
    for i in range(6):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); torch.matmul(a, b); e.record(); torch.cuda.synchronize()
        if i > 0:
            best = min(best, s.elapsed_time(e))
    del a, b
    return 2.0 * n ** 3 / best / 1e9          # flop per ms / 1e9 = TFLOP/s


def timed(torch, fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), ts


def mse_comparison(pkg, steps=10):
    """Test MSE of config 2 after `steps` adaptation steps (the reference's loop: refit after every step)."""
    cands = np.random.default_rng(0).uniform(size=(100000, 2))
    X0 = np.random.RandomState(10).uniform(size=(30, 2))
    Xt = np.random.default_rng(9).uniform(size=(4000, 2))
    Yt = hf_2d(Xt)
    out = {}
    for name, mx in (("CandidateSetMaximizer", pkg.CandidateSetMaximizer(candidates=cands)),
                     ("ALCMaximizer", pkg.ALCMaximizer(candidates=cands, n_reference=1024, seed=0))):
        np.random.seed(0)                          # the fit's restarts draw from NumPy's global stream
        m = pkg.GPDF(2, 0.001, 2, hf_2d, lf_2d, adapt_maximizer=mx)
        m.fit(X0)
        mse0 = m.get_mse(Xt, Yt)
        t0 = time.perf_counter()
        m.adapt(steps, eps=0.0)
        out[name] = {"mse_before": mse0, "mse_after": m.get_mse(Xt, Yt), "steps": len(m.acquired_points),
                     "adapt_s": time.perf_counter() - t0}
        print("mse", name, out[name], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import multifidelity_datafusion_gps_b200 as pkg
    from multifidelity_datafusion_gps_b200 import _ffi, gp
    os.makedirs(args.out, exist_ok=True)
    res = {"card": card(), "reps": args.reps, "dgemm_tflops": dgemm_rate(torch), "shapes": {}}
    print("card", res["card"], "dgemm %.1f TFLOP/s" % res["dgemm_tflops"], flush=True)
    for name, (factory, cands) in shapes(pkg, gp).items():
        m = factory()
        C, npad = int(cands.shape[0]), int(m.hf_model.npad)
        h = _ffi.get_handle(m.device)
        m.acquisition_argmax(cands)                 # warm-up: candidates resident
        argmax_ms, argmax_all = timed(torch, lambda: m.acquisition_argmax(cands), args.reps)
        rows = {}
        for R in (256, 1024, 4096):
            ref = np.random.default_rng(R).uniform(size=(R, cands.shape[1]))
            m.acquisition_alc(cands, ref)           # warm-up: reference rows resident, every kernel paged in
            alc_ms, alc_all = timed(torch, lambda: m.acquisition_alc(cands, ref), args.reps)
            h.profile_enable(True)
            idx, val = m.acquisition_alc(cands, ref)
            prof = {k: {"avg_ms": v[0], "launches": v[1], "what": CLASS_NAMES.get(k)}
                    for k, v in h.profile_read().items() if v[1]}
            h.profile_enable(False)
            rpad = (R + 127) // 128 * 128
            flops = float(C) * npad * npad + 2.0 * C * rpad * npad + float(rpad) * npad * npad
            g_bytes = 16.0 * C * rpad
            rows["R%d" % R] = {
                "alc_ms": alc_ms, "alc_ms_all": alc_all, "alc_over_argmax": alc_ms / argmax_ms,
                "product_flops": flops, "product_tflops_over_call": flops / alc_ms / 1e9,
                "product_rate_vs_dgemm_over_call": flops / alc_ms / 1e9 / res["dgemm_tflops"],
                "g_bytes": g_bytes, "g_hbm_floor_ms": g_bytes / 7.7e9, "g_hbm_floor_share_of_call": g_bytes / 7.7e9 / alc_ms,
                "index": idx, "alc": val, "kernel_classes_one_call": prof}
            gemm = prof.get("gemm")
            if gemm:
                g_ms = gemm["avg_ms"] * gemm["launches"]
                rows["R%d" % R]["g_product_tflops"] = 2.0 * C * rpad * npad / g_ms / 1e9
            print(name, "R=%d" % R, "alc %.2f ms" % alc_ms, "argmax %.2f ms" % argmax_ms,
                  {k: round(v["avg_ms"] * v["launches"], 3) for k, v in prof.items()}, flush=True)
        res["shapes"][name] = {"candidates": C, "N_h": int(m.hf_model.N), "npad": npad, "D": int(m.hf_model.D),
                               "argmax_ms": argmax_ms, "argmax_ms_all": argmax_all, "by_R": rows}
        del m
        gp.release_workspaces()
        torch.cuda.empty_cache()
    res["mse_after_10_steps_config2"] = mse_comparison(pkg)
    with open(os.path.join(args.out, "acq_alc_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
