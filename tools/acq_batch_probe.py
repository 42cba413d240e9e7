"""Greedy batch acquisition against the sequential loop it replaces, on the GPU.

For the three shapes of bench.py's acquisition block (config 2: GPDF 2-D, N_h = 30, 100 000 candidates; config 3:
NARGP 4-D, N_h = 30, 2^20 candidates; bench model: NARGP 4-D, N_h = 1024, N_l = 4096, 2^20 candidates) and
q in {1, 4, 16}: wall time of a resident acquisition_batch(cands, q) against q sequential steps
(acquisition_argmax + the bordered update of _append_hf_point, what adapt does with refit_every > q), each timed
region between device synchronisations after a warm-up; whether both pick the same points; launches per pick; the
per-class kernel times of one batch (mfgp_profile_*: class "argmax" holds the fused update + arg-max kernel); and the
card's name and power limit.  Writes DIR/acq_batch_probe.json.

    python tools/acq_batch_probe.py --out DIR [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def hf_2d(x):                                    # reference tests/test_mfgp_adapt_2d.py:12-14
    x = np.atleast_2d(x)
    return (np.sin(x[:, 0] * 2.2 * np.pi) * np.sin(x[:, 1] * np.pi))[:, None]


def lf_2d(x):                                    # reference tests/test_mfgp_adapt_2d.py:17-19
    x = np.atleast_2d(x)
    return hf_2d(x) - 1.2 * (np.sin(x[:, 0] * np.pi * 0.1) + np.sin(x[:, 1] * np.pi * 0.1))[:, None]


def hf_4d(x):                                    # reference tests/test_mfgp_adapt_4d.py:13-15
    x = np.atleast_2d(x)
    return (np.prod(np.sin(x[:, :4] * np.pi), axis=1) + 5.0)[:, None]


def lf_4d(x):                                    # reference tests/test_mfgp_adapt_4d.py:18-21
    x = np.atleast_2d(x)
    return hf_4d(x) - 0.25 * (np.sin(x[:, 0] * np.pi * 0.1) + np.sin(x[:, 1] * np.pi * 0.05)
                              + np.sin(x[:, 2] * 0.15 * np.pi) + np.sin(x[:, 3] * 0.2 * np.pi))[:, None]


def shapes(pkg, gp):
    """name -> (model factory, candidates), the models of bench.py's acquisition block."""
    rs = np.random.RandomState(10)
    X2, X4 = rs.uniform(size=(30, 2)), rs.uniform(size=(30, 4))

    def config2():
        m = pkg.GPDF(2, 0.001, 2, hf_2d, lf_2d)
        m.fit(X2, theta=np.array([1.2, 0.9, 1e-3]))
        return m

    def config3():
        m = pkg.NARGP(4, hf_4d, lf_4d)
        m.fit(X4, theta=np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 1e-3]))
        return m

    rng = np.random.default_rng(1)                # bench.py workload(1024, 4096, .)
    Xh, Xl = rng.uniform(size=(1024, 4)), rng.uniform(size=(4096, 4))
    yl = lf_4d(Xl)

    def bench_model():
        m = pkg.NARGP(4, hf_4d, None, lf_X=Xl[:8], lf_Y=yl[:8])
        m.lf_X, m.lf_Y = Xl, yl
        m.lf_model = gp.GPRegression(Xl, yl)
        m.lf_model._set_params(np.array([1.0, 0.3, 0.01 * yl.var()]))
        m.fit(Xh, theta=np.array([1.0, 0.3, 1.0, 0.3, 0.1, 0.3, 0.01 * hf_4d(Xh).var()]))
        return m

    c2 = np.random.default_rng(0).uniform(size=(100000, 2))
    c4 = np.random.default_rng(0).uniform(size=(1 << 20, 4))
    return {"config2_gpdf_2d_nh30": (config2, c2), "config3_nargp_4d_nh30": (config3, c4),
            "bench_model_nh1024_nl4096": (bench_model, c4)}


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        out["nvidia_smi"] = None
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
    res = {"card": card(), "reps": args.reps, "shapes": {}}
    for name, (factory, cands) in shapes(pkg, gp).items():
        rows = {}
        base = factory()
        base.acquisition_batch(cands, 16)               # warm-up: candidates resident, every kernel paged in
        h = _ffi.get_handle(base.device)
        for q in (1, 4, 16):
            torch.cuda.synchronize()
            n0 = h.launches
            idx, var = base.acquisition_batch(cands, q)
            launches = h.launches - n0
            ts = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                base.acquisition_batch(cands, q)
                torch.cuda.synchronize()
                ts.append(1e3 * (time.perf_counter() - t0))
            h.profile_enable(True)
            base.acquisition_batch(cands, q)
            prof = {k: {"avg_ms": v[0], "launches": v[1]} for k, v in h.profile_read().items() if v[1]}
            h.profile_enable(False)
            # sequential: q x (arg-max + bordered update) on a fresh copy of the model per repetition
            seq_ts, picks = [], None
            for r in range(args.reps + 1):              # repetition 0 warms the grown shapes up
                m = factory()
                m.acquisition_argmax(cands)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                got = []
                for _ in range(q):
                    j, _ = m.acquisition_argmax(cands)
                    got.append(j)
                    m._append_hf_point(np.vstack([m.hf_X, cands[j]]))
                torch.cuda.synchronize()
                if r:
                    seq_ts.append(1e3 * (time.perf_counter() - t0))
                picks = got
            rows["q%d" % q] = {
                "batch_ms": float(np.median(ts)), "batch_ms_all": ts,
                "sequential_ms": float(np.median(seq_ts)), "sequential_ms_all": seq_ts,
                "speedup": float(np.median(seq_ts) / np.median(ts)),
                "launches_per_pick": launches / q, "picks_equal_sequential": [int(i) for i in idx] == picks,
                "batch_picks": [int(i) for i in idx], "sequential_picks": picks,
                "batch_variances": [float(v) for v in var], "kernel_classes_one_batch": prof}
            print(name, "q=%d" % q, "batch %.2f ms" % rows["q%d" % q]["batch_ms"],
                  "sequential %.2f ms" % rows["q%d" % q]["sequential_ms"],
                  "same picks" if rows["q%d" % q]["picks_equal_sequential"] else "DIFFERENT picks", flush=True)
        res["shapes"][name] = {"candidates": int(cands.shape[0]), "N_h": int(base.hf_model.N),
                               "D": int(base.hf_model.D), "by_q": rows}
        gp.release_workspaces()
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "acq_batch_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
