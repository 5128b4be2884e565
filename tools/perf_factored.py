"""K_ff + dK/dl (UPPER) and K_ef + dK/dl on the S5 packs (or smaller): device time per call (CUDA events, best of
`reps`), device time per kernel (torch.profiler over one call) and bitwise checksums of every output, as one JSON line.
For A/B runs of library builds: GPRB_LIB=variants/libgpr_b200_<name>.so python tools/perf_factored.py [n_struct] [reps].
GPRB_KFF_FACTORED is honoured as set by the caller."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gpr_calculator_b200 import _lib, device as gdev, synthetic as syn   # noqa: E402
from gpr_calculator_b200.SO3 import SO3                                   # noqa: E402

n_struct = int(sys.argv[1]) if len(sys.argv) > 1 else 340
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
E_dev, F_dev = syn.packed_from_batch(SO3(nmax=3, lmax=4, rcut=5.0), [a for a, _, _ in syn.structures(n_struct, 2, 2000)])
e = gdev.Pack(E_dev[0], E_dev[1], E_dev[2])
f = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
NE, NF = e.n_groups, f.n_groups
F64 = torch.float64
K = torch.empty((3 * NF, 3 * NF), dtype=F64, device="cuda")
dK = torch.empty_like(K)
Kef, dKef = (torch.empty((NE, 3 * NF), dtype=F64, device="cuda") for _ in range(2))
Kfe, dKfe = (torch.empty((3 * NF, NE), dtype=F64, device="cuda") for _ in range(2))


def kff():
    _lib.call("gprb_kff", _lib.RBF, f.handle, f.handle, 1.0, 0.1, 2.0, 0, 1e-10, _lib.FF_UPPER, 0, NF,
              gdev.ptr(K), 3 * NF, gdev.ptr(dK), 3 * NF, gdev.stream())


def kef():
    _lib.call("gprb_kef", _lib.RBF, e.handle, f.handle, 1.0, 0.1, 2.0, 0, NF, gdev.ptr(Kef), 3 * NF, gdev.ptr(Kfe), NE,
              gdev.ptr(dKef), 3 * NF, gdev.ptr(dKfe), NE, gdev.stream())


def checksum(M):
    """Sum of the 64-bit patterns (wrapping) and the floating-point sum: equal patterns give equal checksums."""
    return [int(M.view(torch.int64).sum()), float(M.sum())]


def measure(fn, outs):
    fn()                                   # first call: schedules and, on the factored path, the pack's atom plan
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        for name in ("kff_z_kernel", "kff_contract_kernel", "kef_y_kernel", "cov_mma_kernel"):
            if name in ev.key and t > 0:
                kernels[name] = kernels.get(name, 0.0) + t / 1e3
    return {"ms_best": min(times), "ms_all": times, "kernel_ms": kernels, "checksums": [checksum(M) for M in outs]}


res = {"lib": os.path.basename(_lib.LIB_PATH), "GPRB_KFF_FACTORED": os.environ.get("GPRB_KFF_FACTORED"),
       "gpu": torch.cuda.get_device_name(0), "n_struct": n_struct, "NE": NE, "NF": NF,
       "kff_upper": measure(kff, (K, dK)), "kef": measure(kef, (Kef, Kfe, dKef, dKfe))}
res["kef_transposed_bitwise"] = bool(torch.equal(Kef, Kfe.T) and torch.equal(dKef, dKfe.T))
print(json.dumps(res))
