"""Tuning aid: per-CTA cycle breakdown of k_select_hot on the bench workload.  Needs a library built with the
statistics compiled in (they are NOT in the production build):
    CNB_NVCC_DEFINES=-DCNB_SELECT_STATS python centernet_b200/build.py --force && python tools/select_stats.py"""
import ctypes
import os
import sys

import numpy as np
import torch

sys.path.insert(0, '.')
from centernet_b200 import decode as D
import centernet_b200

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
g = torch.Generator(device='cuda').manual_seed(317)
bat = []
for i in range(3):
    bat.append((torch.sigmoid(torch.randn(B, 80, 128, 128, device='cuda', generator=g) - 2.19),
                torch.rand(B, 2, 128, 128, device='cuda', generator=g) * 32, torch.rand(B, 2, 128, 128, device='cuda', generator=g)))
for i in range(6):
    D.ctdet_decode(bat[i % 3][0], bat[i % 3][1], reg=bat[i % 3][2], K=100)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(60):
    D.ctdet_decode(bat[i % 3][0], bat[i % 3][1], reg=bat[i % 3][2], K=100)
e1.record(); torch.cuda.synchronize()
print("B=%d wb=%s: %.4f ms per call" % (B, os.environ.get("CNB_SELECT_WB", "default"), e0.elapsed_time(e1) / 60))
lib = ctypes.CDLL(os.path.join(os.path.dirname(centernet_b200.__file__), "lib", "libcenternet_b200.so"))
n = 148
full = np.zeros((192, 10), np.uint64)
assert lib.cnb_debug_select_stats(full.ctypes.data_as(ctypes.c_void_p), 192) == 0
out = full[:n]
print("finalize phases of image 7 [loads+sync, take, cut+sort, fill, emit] cycles, survivors, segments:", [int(v) for v in full[191, :7]])
o = out.astype(np.float64)
names = ["total", "wait", "boot", "flush", "fin_cyc", "units", "n_boot", "n_flush", "n_fin", "smid"]
print("mean", {k: round(float(o[:, i].mean()), 1) for i, k in enumerate(names)})
print("max total %d min %d" % (o[:, 0].max(), o[:, 0].min()))
order = np.argsort(-o[:, 0])
for r in list(order[:12]) + list(order[-6:]):
    print("cta %3d" % r, {k: int(o[r, i]) for i, k in enumerate(names)})
# least squares: total ~ a*units + b*n_boot + c*n_flush + d*n_fin
A = np.stack([o[:, 5], o[:, 6], o[:, 7], o[:, 8], np.ones(n)], 1)
coef, *_ = np.linalg.lstsq(A, o[:, 0], rcond=None)
print("fit total = %.0f*units + %.0f*boot + %.0f*flush + %.0f*fin + %.0f" % tuple(coef))
print("per-plane steady: (total - boot - flush)/units =", round(float(((o[:, 0] - o[:, 2] - o[:, 3]) / o[:, 5]).mean()), 1),
      " wait/unit =", round(float((o[:, 1] / o[:, 5]).mean()), 1))
