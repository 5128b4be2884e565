"""Total stress of batches of structures against the per-atom stress route, on the S5 training set (340 x Cu32,
N = 32 980): structures per second of GP.predict_structures(stress=True, return_std=True) (one row per atom, E / F / S
and their sigma) and of a loop of GP.predict_structure(stress=True, return_std=True) (6 rows per atom, E / F sigma only),
plus the device time of gprb_virial_rows on one batch.

    python tools/perf_stress.py [n_train] [n_test] [batch] [reps]      (defaults 340 64 32 3)

Prints one JSON line with the GPU's name and power limit next to the numbers, and the largest |S_batched - sum_a S_atom|
relative to max |S| over the test set."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gpr_calculator_b200 import _lib, device as gdev, synthetic as syn   # noqa: E402
from gpr_calculator_b200.SO3 import SO3                                   # noqa: E402
from gpr_calculator_b200.gaussianprocess import GP                        # noqa: E402
from gpr_calculator_b200.kernels import RBF_mb                            # noqa: E402

n_train = int(sys.argv[1]) if len(sys.argv) > 1 else 340
n_test = int(sys.argv[2]) if len(sys.argv) > 2 else 64
batch = int(sys.argv[3]) if len(sys.argv) > 3 else 32
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3

des = SO3(nmax=3, lmax=4, rcut=5.0, stress=True)
labelled = syn.structures(n_train, 2, 2000)
E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
y = syn.targets(labelled)
gp = GP(kernel=RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
gp.train_x = {"energy": gdev.Pack(E_dev[0], E_dev[1], E_dev[2]), "force": gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])}
gp.train_y = {"energy": list(y[:n_train, 0]), "force": y[n_train:, 0].reshape(-1, 3)}
gp.N_energy, gp.N_forces = n_train, gp.train_x["force"].n_groups
gp.fit(opt=False, show=False)
tests_ = [a for a, _, _ in syn.structures(n_test, 2, 3000)]


def timed(fn):
    fn()                                  # warm-up: modules, cuBLAS algorithms, the explicit inverse of the small-m route
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best, out


t_batched, batched = timed(lambda: gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=batch, stress=True))
t_loop, loop = timed(lambda: [gp.predict_structure(s_, stress=True, return_std=True, f_tol=1e-12) for s_ in tests_])
S_b = np.array([t[2] for t in batched])
S_l = np.array([t[2].sum(axis=0) for t in loop])

# gprb_virial_rows alone on one batch: HBM bytes it must read (8 * 9 * d per seq row) over device time
r = des.calculate_batch(tests_[:batch], to_host=False)
d, n_seq, A = r["x"].shape[1], r["rdxdr"].shape[0], r["x"].shape[0]
V = torch.empty((A, d, 6), dtype=torch.float64, device="cuda")
n_launch = 200
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for it in range(2):
    e0.record()
    for _ in range(n_launch):
        _lib.call("gprb_virial_rows", A, d, gdev.ptr(r["seq_ptr"]), gdev.ptr(r["rdxdr"]), gdev.ptr(V), gdev.stream())
    e1.record()
    torch.cuda.synchronize()
k_us = e0.elapsed_time(e1) * 1e3 / n_launch

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                     text=True).stdout.strip().splitlines()
print(json.dumps({"gpu": gpu[torch.cuda.current_device()] if gpu else torch.cuda.get_device_name(),
                  "n_train": n_train, "N": int(gp.alpha_.shape[0]), "n_test": n_test, "batch": batch,
                  "batched_structs_per_s": n_test / t_batched, "loop_structs_per_s": n_test / t_loop,
                  "speedup": t_loop / t_batched,
                  "max_rel_diff_S": float(np.abs(S_b - S_l).max() / np.abs(S_l).max()),
                  "virial_rows": {"atoms": A, "seq_rows": n_seq, "d": d, "us": k_us,
                                  "GB_per_s": 8 * 9 * d * n_seq / (k_us * 1e-6) * 1e-9}}))
