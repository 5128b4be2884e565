"""Quick device timing of gprb_kff on random packed rows shaped like the S5 config (dev tool)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from gpr_calculator_b200 import _lib
from gpr_calculator_b200.device import Pack, empty, ptr, stream, c_vp

def run(NF, rows_lo, rows_hi, d=30, grad=False, mode=_lib.FF_FULL, kernel=_lib.RBF, reps=3):
    rng = np.random.default_rng(0)
    ind = rng.integers(rows_lo, rows_hi + 1, size=NF)
    R = int(ind.sum())
    x = torch.rand(R, d, dtype=torch.float64, device='cuda') + 0.5
    dx = torch.randn(R, d, 3, dtype=torch.float64, device='cuda')
    ele = torch.full((R,), 29, dtype=torch.int32, device='cuda')
    p = Pack(x, ele, ind, dxdr=dx)
    K = empty(3 * NF, 3 * NF); dK = empty(3 * NF, 3 * NF) if grad else None
    pairs = p.pair_count(p)
    if mode == _lib.FF_SYMMETRIC:
        pairs_eval = None
    def go():
        _lib.call("gprb_kff", kernel, p.handle, p.handle, 1.0, 0.5, 2.0, 0 if grad else 1, 1e-10, mode, 0, NF,
                  ptr(K), 3 * NF, ptr(dK), 3 * NF, stream())
    go(); torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); go(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    fl = 32 * d * pairs
    print(json.dumps({"NF": NF, "rows": R, "grad": grad, "mode": mode, "kernel": kernel, "ms": best, "pairs": pairs,
                      "ps_per_pair": best * 1e9 / pairs, "alg_tflops_fullblock": fl / best * 1e-9}))

run(1000, 24, 33)
run(4000, 24, 33)
run(4000, 24, 33, grad=True)
run(4000, 24, 33, mode=_lib.FF_SYMMETRIC)
run(4000, 32, 32)
run(2000, 40, 48)
run(4000, 24, 33, kernel=_lib.DOT)
