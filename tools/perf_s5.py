"""K_ff(+grad) kernel on the real S5 (or smaller) packs: device time, algorithmic TFLOP/s and checksums of K / dK/dl
(for A/B runs of library variants: GPRB_LIB=variants/libgpr_b200_<name>.so python tools/perf_s5.py [n_struct] [grad] [reps])."""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gpr_calculator_b200 import _lib, device as gdev, synthetic as syn   # noqa: E402
from gpr_calculator_b200.SO3 import SO3                                   # noqa: E402

n_struct = int(sys.argv[1]) if len(sys.argv) > 1 else 340
grad = int(sys.argv[2]) if len(sys.argv) > 2 else 1
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 2
mode = int(sys.argv[4]) if len(sys.argv) > 4 else _lib.FF_UPPER
des = SO3(nmax=3, lmax=4, rcut=5.0)
E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in syn.structures(n_struct, 2, 2000)])
f = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
NF = f.n_groups
pairs = syn.pair_counts(F_dev[2].cpu().numpy(), F_dev[3], symmetric=(mode != _lib.FF_FULL))
K = torch.empty((3 * NF, 3 * NF), dtype=torch.float64, device="cuda")
dK = torch.empty((3 * NF, 3 * NF), dtype=torch.float64, device="cuda") if grad else None


def go():
    _lib.call("gprb_kff", _lib.RBF, f.handle, f.handle, 1.0, 0.1, 2.0, 0 if grad else 1, 1e-10, mode, 0, NF,
              gdev.ptr(K), 3 * NF, gdev.ptr(dK), 3 * NF, gdev.stream())


t0 = time.time()
go()                      # first call: row schedule and, on the factored path, the pack's atom plan
torch.cuda.synchronize()
first_ms = (time.time() - t0) * 1e3
best = 1e30
for _ in range(reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    go()
    e1.record()
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1))
peak = np.zeros(1)
_lib.call("gprb_fp64_dmma_peak", peak.ctypes.data, gdev.stream())
tf = 32 * 30 * pairs / best * 1e-9
print(json.dumps({"lib": os.path.basename(_lib.LIB_PATH), "GPRB_KFF_FACTORED": os.environ.get("GPRB_KFF_FACTORED"),
                  "first_ms": first_ms, "n_struct": n_struct, "NF": NF, "grad": grad, "mode": mode, "ms": best,
                  "tflops": tf, "peak": float(peak[0]), "frac": tf / float(peak[0]),
                  "sumK": float(K.sum()), "sum_absK": float(K.abs().sum()),
                  "sumdK": float(dK.sum()) if grad else None, "sum_absdK": float(dK.abs().sum()) if grad else None}))
