"""Times one MC sweep at a small high-fidelity level (default N_h = 30, N_l = 100, M = 2^20, S = 100) and prints a
fingerprint of the result.  MFGP_PROBE_SAVE=<file.npy> keeps the result and MFGP_PROBE_COMPARE=<file.npy> compares
with a kept one, so that two builds of the library (MFGP_LIB) can be set against each other."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import multifidelity_datafusion_gps_b200 as pkg  # noqa: E402
from multifidelity_datafusion_gps_b200 import gp  # noqa: E402

nh = int(sys.argv[1]) if len(sys.argv) > 1 else 30
nl = int(sys.argv[2]) if len(sys.argv) > 2 else 100
m = int(sys.argv[3]) if len(sys.argv) > 3 else 32 ** 4
S = int(sys.argv[4]) if len(sys.argv) > 4 else 100
wl = bench.workload(nh, nl, m)
model = bench.build_model(pkg, gp, wl)
dX, dw = gp.to_device(wl["Xt"], model.device), gp.to_device(wl["w"], model.device)
model.predict_mc_device(dX[:256], S, None, 2, 0, dw[:256])
torch.cuda.synchronize()
for rep in range(3):
    s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_ev.record()
    mean, var, wsum = model.predict_mc_device(dX, S, None, 2, 0, dw)
    e_ev.record(); torch.cuda.synchronize()
    ms = s_ev.elapsed_time(e_ev)
    print("N_h=%d N_l=%d M=%d S=%d rep %d: %.2f ms  %.1f M samples/s  pce_mean=%.15g  sum(var)=%.15g" %
          (nh, nl, m, S, rep, ms, m * S / ms / 1e3, wsum, float(var.sum().item())))
out = os.environ.get("MFGP_PROBE_SAVE")
if out:
    np.save(out, np.stack([mean.cpu().numpy(), var.cpu().numpy()]))
cmp = os.environ.get("MFGP_PROBE_COMPARE")
if cmp:
    ref = np.load(cmp)
    cur = np.stack([mean.cpu().numpy(), var.cpu().numpy()])
    print("vs %s: max |d mean| = %.3e (rel %.3e), max |d var| = %.3e" %
          (cmp, np.abs(cur[0] - ref[0]).max(), np.abs(cur[0] - ref[0]).max() / np.abs(ref[0]).max(),
           np.abs(cur[1] - ref[1]).max()))
