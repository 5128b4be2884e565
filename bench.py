#!/usr/bin/env python
"""Benchmark of the covariance hot path (BASELINE.json metric: K_ff/K_ef build GFLOP/s, K-build wall time,
E/F predictions per second) on 1..8 B200.

    python bench.py --gpus N --steps K --warmup W              # this framework (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU implementation (rank 0 only)

Workload (config.workload, SURVEY.md §8d S5 = BASELINE.json configs[4], the scale-out configuration, which
fits one GPU): 340 synthetic Cu fcc 2x2x2 structures (32 atoms), SO3(nmax=3, lmax=4, rcut=5.0) computed on
the device, every atom a force centre: N = 340 energy rows + 32 640 force rows, RBF zeta = 2,
(sigma, l) = (1.0, 0.1), noise 0.002 / 0.1.

A step = one likelihood-loop covariance build: K and dK/dl of the training set (K_ee, K_ef/K_fe, K_ff
with the gradient epilogue, gaussianprocess.py:158-159 -> RBF_mb.k_total_with_grad), rows block-sharded
over the ranks, K all-gathered over NCCL and mirrored (strong scaling: the total work is fixed).
  value  : algorithmic GFLOP/s = (32 d P_ff + 8 d P_ef + 2 d P_ee) / step time, P = same-species atom pairs
           actually evaluated (the symmetric build evaluates the J >= I blocks only), operands resident in HBM.
  e2e    : the same flops over the time of one GP.log_marginal_likelihood(theta, eval_gradient=True)
           call starting from HOST (pinned) packed arrays: H2D + row packing + K/dK build + cuSOLVER
           potrf/potrs + inverse rows (trailing-block potrs) + gradient trace + D2H of the reduced scalars.
  roofline: K_ff kernel alone (CUDA events around gprb_kff on its stream) against the FP64 tensor (DMMA)
           peak measured live by gprb_fp64_dmma_peak (MEASURED_PEAKS.json carries no fp64 entry).
  cpu_baseline: the UNMODIFIED reference C++ (oracle/_ref) on a bounded sample of the same workload,
           row-split over the host cores like the reference's MPI split.

--dump-outputs DIR writes what the timed calls returned in their last step as DIR/<name>.npy (float64), so that two
builds can be compared output by output on identical (seeded) inputs: a fixed sample of K and dK/dl (rows = columns =
K_sample_index), the LML and its gradient of the end-to-end leg, and the predictions of a fixed sample of structures.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

D = 30
SIGMA, ELL, ZETA = 1.0, 0.1, 2.0
NOISE_E, NOISE_F = 0.002, 0.1
WORKLOADS = {
    # name: (structures, fcc repeats, seed0, description)
    "s5": (340, 2, 2000, "S5: 340 x Cu fcc 32 atoms, all atoms force centres, N = 340 E + 32640 F rows"),
    "s4": (200, 3, 1000, "S4: 200 x Cu fcc 108 atoms, all atoms force centres, N = 200 E + 64800 F rows"),
    "medium": (100, 2, 2000, "100 x Cu fcc 32 atoms (profiling size), N = 100 E + 9600 F rows"),
    "small": (24, 2, 2000, "24 x Cu fcc 32 atoms (development size)"),
}


# DRAM bytes per launch of the K_ff(+grad) kernel, from ncu (13.82 GB read + 17.18 GB written at S5)
KFF_DRAM_TRAFFIC = {"s5": 30.995e9}


SO3_CPU_SECONDS = []     # numpy port of SO3.calculate (oracle/so3.py), seconds per structure of the CPU sample


def flops_of(p_ff, p_ef, p_ee, d=D):
    return 32.0 * d * p_ff + 8.0 * d * p_ef + 2.0 * d * p_ee


# --dump-outputs: K and dK/dl of S5 are 77 GB each, so a fixed sample of rows (= columns) is written (about 20 MB in all)
DUMP_K_ROWS, DUMP_K_ENERGY_ROWS, DUMP_STRUCTURES = 1024, 128, 1024


def k_sample_index(NE, N):
    """Sorted, seeded row (= column) indices of the N x N covariance: up to DUMP_K_ENERGY_ROWS energy rows, the rest
    force rows, so that the sample holds parts of the EE, EF and FF blocks and their diagonals."""
    rng = np.random.default_rng(0)
    n_e = min(NE, DUMP_K_ENERGY_ROWS)
    n_f = min(N - NE, DUMP_K_ROWS - n_e)
    return np.sort(np.concatenate([rng.choice(NE, n_e, replace=False), NE + rng.choice(N - NE, n_f, replace=False)]))


def dump(dir_, name, a):
    if dir_ is not None:
        os.makedirs(dir_, exist_ok=True)
        np.save(os.path.join(dir_, name + ".npy"), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def summary(self, t0, t1):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [v.strip() for v in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: unmodified reference C++ (oracle/_ref), row-split over host threads
# ------------------------------------------------------------------------------------------------
def cpu_sample(n_struct, nrep, seed0):
    """Host packed training data of the first `n_struct` structures of the workload (device SO3 when a
    GPU is present is NOT used here: the sample is produced by the numpy oracle descriptor so that the
    reference arm runs without touching the product)."""
    from oracle import so3 as oso3
    from gpr_calculator_b200.synthetic import cu_fcc
    e_items, f_items = [], []
    global SO3_CPU_SECONDS
    for k in range(n_struct):
        at, _, _ = cu_fcc(nrep, seed0 + k)
        t0 = time.perf_counter()
        x, dxdr, seq = oso3.so3_calculate(at.positions, at.cell, at.pbc, at.numbers, 3, 4, 5.0, 2.0)
        SO3_CPU_SECONDS.append(time.perf_counter() - t0)
        ele = np.asarray(at.numbers, dtype=np.int32)
        e_items.append((x, ele))
        for i in range(len(at)):
            ids = np.flatnonzero(seq[:, 1] == i)
            f_items.append((x[seq[ids, 0]], dxdr[ids], ele[seq[ids, 0]]))
    return e_items, f_items


def reference_build(e_items, f_items, threads):
    """K and dK/dl blocks with grad, the way RBF_mb.k_total_with_grad assembles them (RBF_mb.py:173-204),
    each block row-split over `threads` workers like the MPI split (RBF_mb.py:257-301, 348-431, 471-481)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import kernels as ok
    O = ok.RBFOracle("ref" if ok.have_ref() else "port")
    E, F = ok.list_to_tuple(e_items, mode="energy"), ok.list_to_tuple(f_items)

    def chunks(items):
        n = len(items)
        per = max(1, -(-n // threads))
        return [items[i:i + per] for i in range(0, n, per)]

    with ThreadPoolExecutor(max_workers=threads) as pool:
        ff = list(pool.map(lambda c: O.kff_C(ok.list_to_tuple(c), F, SIGMA, ELL, ZETA, grad=True), chunks(f_items)))
        fe = list(pool.map(lambda c: O.kef_C(E, ok.list_to_tuple(c), SIGMA, ELL, ZETA, grad=True), chunks(f_items)))
        ee = list(pool.map(lambda c: O.kee_C(ok.list_to_tuple(c, mode="energy"), E, SIGMA, ELL, ZETA, grad=True), chunks(e_items)))
    out = []
    for k in (0, 2):          # K and dK/dl (the wrappers return (K, dK/dsigma, dK/dl))
        Kff = np.vstack([b[k] for b in ff])
        Kef = np.hstack([b[k] for b in fe])
        Kee = np.vstack([b[k] for b in ee])
        out.append(np.block([[Kee, Kef], [Kef.T, Kff]]))
    return out[0], out[1]


def sample_pairs(e_items, f_items):
    re_ = sum(len(x) for x, _ in e_items)
    rf = sum(len(x) for x, _, _ in f_items)
    return rf * rf, re_ * rf, re_ * re_    # single species: every row pair counts; full rectangular blocks


def run_cpu(n_struct, nrep, seed0, steps, warmup, threads):
    from oracle import kernels as ok
    ok.build(ref=os.path.isdir("/root/reference"), port=True)
    e_items, f_items = cpu_sample(n_struct, nrep, seed0)
    fl = flops_of(*sample_pairs(e_items, f_items))
    last = None
    for _ in range(warmup):
        reference_build(e_items, f_items, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        last = reference_build(e_items, f_items, threads)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    kind = "reference" if ok.have_ref() else "port"
    sample = ("first %d structures of the workload (%d E + %d F centres, %.3g K_ff pairs), K and dK/dl "
              "(rbf_k*_many_with_grad)" % (n_struct, len(e_items), len(f_items), sample_pairs(e_items, f_items)[0]))
    return fl / dt * 1e-9, dt, kind, sample, (e_items, f_items, last)


PARITY_TOL = 1e-10


def parity_vs_reference(e_items, f_items, K_ref, dK_ref, atoms_list):
    """The CUDA path on the SAME host descriptors as the CPU leg (real Cu32 rows: cos-similarity 0.998..1, |x| ~ 7e3,
    l = 0.1) against the K / dK/dl the reference C++ just produced (rbf_kernel.cpp:5-98, 101-253, 475-640).
    Two measures per matrix: per entry against the Cauchy-Schwarz scale sqrt(K_ii K_jj) of that entry (for dK/dl times
    the bound (1/l^3 + 2/l) of |dlog k/dl|), and against the largest entry of its block (EE, EF, FF)."""
    import torch
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.utilities import list_to_tuple
    data = {"energy": list_to_tuple(e_items, mode="energy"), "force": list_to_tuple(f_items)}
    K, dK = RBF_mb(para=[SIGMA, ELL], zeta=ZETA).k_total_device(data, None, grad=True)
    K, dK = K.cpu().numpy(), dK.cpu().numpy()
    NE = len(e_items)
    d = np.sqrt(np.abs(np.diag(K_ref)))
    cs = np.outer(d, d)
    out = {"max_rel_K": float((np.abs(K - K_ref) / cs).max()),
           "max_rel_dK": float((np.abs(dK - dK_ref) / (cs * (1.0 / ELL ** 3 + 2.0 / ELL))).max())}
    blocks = {"ee": (slice(0, NE), slice(0, NE)), "ef": (slice(0, NE), slice(NE, None)), "ff": (slice(NE, None), slice(NE, None))}
    for name, (r, c) in blocks.items():
        out["block_rel_K_" + name] = float(np.abs(K[r, c] - K_ref[r, c]).max() / np.abs(K_ref[r, c]).max())
        out["block_rel_dK_" + name] = float(np.abs(dK[r, c] - dK_ref[r, c]).max() / np.abs(dK_ref[r, c]).max())
    # descriptor producer on the same structures: device SO3 against the numpy restatement the CPU leg used
    from gpr_calculator_b200.SO3 import SO3
    r = SO3(nmax=3, lmax=4, rcut=5.0).calculate_batch(atoms_list, to_host=False)
    x_dev = r["x"].cpu().numpy()
    x_ref = np.concatenate([x for x, _ in e_items])
    out["so3_max_rel_x"] = float(np.abs(x_dev - x_ref).max() / np.abs(x_ref).max())
    out.update({"n": int(K_ref.shape[0]), "tol": PARITY_TOL,
                "reference": "oracle/_ref (unmodified rbf_kernel.cpp) on the first %d structures, same host descriptors" % len(e_items)})
    worst = max(v for k, v in out.items() if k.startswith(("max_rel", "block_rel")))
    out["passed"] = bool(worst <= PARITY_TOL)
    return out


def sharded_parity(des, nrep, seed0, n_struct=24):
    """Multi-GPU parity before anything is timed: the row-sharded build (fused peer gather or NCCL gather) of a small
    workload against the window-free build of the same packs on this rank; LML and gradient against an unsharded
    evaluation of the same algebra (every rank evaluates; the caller reduces with MAX)."""
    import torch
    from gpr_calculator_b200 import device as gdev, dist as gdist, synthetic as syn
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    labelled = syn.structures(n_struct, nrep, seed0)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
    e = gdev.Pack(E_dev[0], E_dev[1], E_dev[2])
    f = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
    gp = GP(kernel=RBF_mb(para=[SIGMA, ELL], zeta=ZETA), descriptor=des, noise_e=NOISE_E, noise_f=NOISE_F, log_file=None)
    gp.train_x = {"energy": e, "force": f}
    gp.y_train = syn.targets(labelled)
    K1, dK1 = gp.kernel.k_total_device(gp.train_x, None, grad=True)
    NE, N = e.n_groups, K1.shape[0]
    errK = errdK = 0.0
    for _ in range(2):                        # the second build re-uses (and re-zeroes) the peer-mapped matrix
        K, dK, ranges = gp._build_K(grad=True)
        errK = max(errK, float((K - K1).abs().max() / K1.abs().max()))
        off = 0
        cols = torch.arange(N, device="cuda")
        for (r0, r1) in ranges:
            if r1 > r0:
                rows, ref = dK[off:off + (r1 - r0)], dK1[r0:r1]
                rr = torch.arange(r0, r1, device="cuda")
                if r1 <= NE:
                    mask = (cols[None, :] < NE).expand(r1 - r0, N)
                else:
                    mask = (cols[None, :] < NE) | (((cols[None, :] - NE) // 3) >= ((rr[:, None] - NE) // 3))
                errdK = max(errdK, float(((rows - ref).abs() * mask).max() / dK1.abs().max()))
            off += r1 - r0
    theta = np.array([SIGMA, ELL])
    lml, grad = gp.log_marginal_likelihood(theta, eval_gradient=True)
    # the same evaluation without sharding: this rank's window-free K / dK through the same entry point
    alpha, out = gp._lml_eval(K1.clone(), dK1, [(0, N)], NOISE_E, NOISE_F, want_grad=True)
    lml1 = -0.5 * out[1] - out[0] - N / 2 * np.log(2 * np.pi)
    g1 = np.array([((out[1] - N) - 2.0 * out[3]) / SIGMA, out[2]])
    gp.release_peer()
    return {"max_rel_K": errK, "max_rel_dK": errdK, "lml_rel": abs(lml - lml1) / abs(lml1),
            "grad_rel": float(np.abs(grad - g1).max() / np.abs(g1).max()), "N": int(N),
            "gather": "peer" if gdist.peer_gather_enabled() else "nccl"}


def _median_ms(fn, reps):
    import torch
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def small_n_block(des):
    """Per-step retrain latency at the sizes of BASELINE configs 1-3 (on-the-fly runs: N = 50 ... 770).
    c1a / c1b: Cu32 synthetic sets (2 E + 16 F centres = 50 rows, 4 E + 56 F = 172 rows); c2: the reference's real
    Pd4/MgO training set (tests/golden/pd4.npz = examples/database/pd4-RBF.db: 155 E x 220 atoms, three species, + 205 F
    centres = 770 rows, 34 100 stacked energy rows) with its stored hyper-parameters."""
    import contextlib
    import io
    import tempfile
    import torch
    from gpr_calculator_b200 import _lib, asedb, synthetic as syn
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.utilities import SimpleAtoms
    out = {}

    def measure(gp, theta, probe_atoms, tag, what):
        lml = lambda: gp.log_marginal_likelihood(theta, eval_gradient=True)     # noqa: E731
        lml()
        lml()
        ms_lml = _median_ms(lml, 15)
        _lib.PROFILE = []
        lml()
        torch.cuda.synchronize()
        prof, _lib.PROFILE = _lib.PROFILE, None
        parts = {}
        for n, a, b, h in prof:
            parts[n] = round(parts.get(n, 0.0) + a.elapsed_time(b), 4)
        with contextlib.redirect_stdout(io.StringIO()):
            gp.kernel.update(list(theta))
            gp.fit(opt=True, show=False, maxiter=10)
            gp.kernel.update(list(theta))
            t0 = time.perf_counter()
            gp.fit(opt=True, show=False, maxiter=10)
            torch.cuda.synchronize()
            ms_fit = (time.perf_counter() - t0) * 1e3
        pred = lambda: gp.predict_structure(probe_atoms, stress=False, return_std=True)   # noqa: E731
        pred()
        pred()
        ms_pred = _median_ms(pred, 15)
        out[tag] = {"workload": what, "N": int(len(gp.y_train)), "lml_grad_ms": ms_lml, "fit_maxiter10_ms": ms_fit,
                    "predict_structure_ms": ms_pred, "lml_device_ms_by_entry_point": parts}

    for tag, n_s, centres in (("c1_n50", 2, 8), ("c1_n172", 4, 14)):
        labelled = syn.structures(n_s, 2, 2000)
        E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled], centres_per_structure=centres)
        E_h, _k1 = syn.to_host(E_dev)
        F_h, _k2 = syn.to_host(F_dev)
        gp = GP(kernel=RBF_mb(para=[SIGMA, ELL], zeta=ZETA), descriptor=des, noise_e=NOISE_E, noise_f=NOISE_F, log_file=None)
        gp.train_x = {"energy": E_h, "force": F_h}
        y = syn.targets(labelled, centres_per_structure=centres)
        gp.train_y = {"energy": list(y[:n_s, 0]), "force": y[n_s:, 0].reshape(-1, 3)}
        gp.update_y_train()
        gp.N_energy, gp.N_forces = n_s, n_s * centres
        measure(gp, np.array([SIGMA, ELL]), syn.cu_fcc(2, 5000)[0], tag,
                "%d Cu32 structures: %d E + %d F centres" % (n_s, n_s, n_s * centres))
    path = os.path.join(ROOT, "tests", "golden", "pd4.npz")
    if os.path.exists(path):
        g = np.load(path)
        with tempfile.TemporaryDirectory() as tmp:
            rows = []
            for k in range(len(g["energy"])):
                at = SimpleAtoms(g["numbers"], g["positions"][k], g["cell"], g["pbc"])
                f_in = g["force_in"][g["force_in_ptr"][k]:g["force_in_ptr"][k + 1]]
                rows.append((at, {"dft_energy": float(g["dft_energy"][k]), "dft_fmax": float(np.abs(g["force"][k]).max())},
                             {"energy": float(g["energy"][k]), "force": g["force"][k], "energy_in": bool(g["energy_in"][k]),
                              "force_in": [int(i) for i in f_in]}))
            db, js = os.path.join(tmp, "pd4.db"), os.path.join(tmp, "pd4.json")
            asedb.write_rows(db, rows)
            model = json.loads(str(g["model_json"]))
            model["db_filename"] = db
            with open(js, "w") as fp:
                json.dump(model, fp)
            # GP.load opens the default log file gpr.log in the working directory: keep it in the temporary one
            with contextlib.redirect_stdout(io.StringIO()), contextlib.chdir(tmp):
                gp = GP.load(js)
        gp.log_file = None
        theta = np.array(gp.kernel.parameters())
        measure(gp, theta, SimpleAtoms(g["numbers"], g["positions"][-1], g["cell"], g["pbc"]), "c2_pd4",
                "Pd4/MgO fixture of the reference (examples/database/pd4-RBF.db): 155 E x 220 atoms (Mg/O/Pd) + 205 F centres")
        e_rows = int(gp.train_x["energy"][0].shape[0])
        kee_ms = out["c2_pd4"]["lml_device_ms_by_entry_point"].get("gprb_kee", 0.0)
        if kee_ms > 0:
            pairs = sum(int((gp.train_x["energy"][1] == z).sum()) ** 2 for z in np.unique(gp.train_x["energy"][1]))
            out["c2_pd4"]["kee"] = {"energy_rows": e_rows, "same_species_pairs": pairs, "ms": kee_ms,
                                    "tflops": 2.0 * gp.train_x["energy"][0].shape[1] * pairs / kee_ms * 1e-9,
                                    "flop_per_pair": "2 d (K_ee with dK/dl, rbf_kernel.cpp:5-98)"}
    return out


def s4_block(des, maxiter, budget_s):
    """BASELINE config 4: 200 x Cu fcc 108 atoms (N = 65 000): one K + dK/dl build and one GP.fit(opt=True, maxiter)."""
    import contextlib
    import io
    import torch
    from gpr_calculator_b200 import _lib, device as gdev, synthetic as syn
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    n_struct, nrep, seed0, desc = WORKLOADS["s4"]
    labelled = syn.structures(n_struct, nrep, seed0)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled], chunk=16)
    e_pack = gdev.Pack(E_dev[0], E_dev[1], E_dev[2])
    f_pack = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
    p_ff = syn.pair_counts(F_dev[2].cpu().numpy(), F_dev[3], symmetric=True)
    p_ee = syn.pair_counts(E_dev[1].cpu().numpy(), E_dev[2], symmetric=False)
    p_ef = e_pack.pair_count(f_pack)
    N = e_pack.n_groups + 3 * f_pack.n_groups
    del E_dev, F_dev
    gp = GP(kernel=RBF_mb(para=[SIGMA, ELL], zeta=ZETA), descriptor=des, noise_e=NOISE_E, noise_f=NOISE_F, log_file=None)
    gp.train_x = {"energy": e_pack, "force": f_pack}
    y = syn.targets(labelled)
    gp.train_y = {"energy": list(y[:n_struct, 0]), "force": y[n_struct:, 0].reshape(-1, 3)}
    gp.update_y_train()
    gp.N_energy, gp.N_forces = e_pack.n_groups, f_pack.n_groups
    out = gp._build_K(grad=True)       # warm-up
    del out
    torch.cuda.synchronize()
    _lib.PROFILE = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    out = gp._build_K(grad=True)
    ev1.record()
    torch.cuda.synchronize()
    del out
    prof, _lib.PROFILE = _lib.PROFILE, None
    ms = ev0.elapsed_time(ev1)
    kff_ms = sum(a.elapsed_time(b) for n, a, b, _ in prof if n == "gprb_kff")
    peak = np.zeros(1)
    _lib.call("gprb_fp64_dmma_peak", peak.ctypes.data, gdev.stream())
    res = {"workload": desc, "N": int(N), "k_build_ms": ms, "gflops": flops_of(p_ff, p_ef, p_ee) / ms * 1e-6,
           "kff_ms": kff_ms, "kff_frac_of_dmma_peak": 32.0 * D * p_ff / (kff_ms * 1e-3) * 1e-12 / float(peak[0])}
    # one full GP.fit(opt=True, maxiter) from the default hyper-parameters; a wall budget stops a long optimisation
    evals, t_start = [], time.perf_counter()
    orig = gp.log_marginal_likelihood

    class _Budget(Exception):
        pass

    def counted(params, eval_gradient=False, clone_kernel=False):
        if evals and time.perf_counter() - t_start > budget_s:
            raise _Budget()
        t0 = time.perf_counter()
        r = orig(params, eval_gradient=eval_gradient, clone_kernel=clone_kernel)
        torch.cuda.synchronize()
        evals.append(time.perf_counter() - t0)
        return r

    gp.log_marginal_likelihood = counted
    stopped = False
    with contextlib.redirect_stdout(io.StringIO()):
        try:
            gp.fit(opt=True, show=False, maxiter=maxiter)
        except _Budget:
            stopped = True
    torch.cuda.synchronize()
    res["fit"] = {"call": "GP.fit(opt=True, maxiter=%d)" % maxiter, "wall_s": time.perf_counter() - t_start,
                  "lml_evaluations": len(evals), "s_per_lml_evaluation": float(np.mean(evals)) if evals else None,
                  "stopped_by_wall_budget": stopped, "budget_s": budget_s,
                  "theta": [float(v) for v in gp.kernel.parameters()]}
    return res


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="s5", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-structures", type=int, default=None, help="structures in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--predict-structures", type=int, default=10000, help="test structures of the prediction leg")
    ap.add_argument("--predict-batch", type=int, default=128,
                    help="structures per device pass of GP.predict_structures (measured at S5: 82.9 / 84.1 / 85.1 structures/s for 32 / 64 / 128)")
    ap.add_argument("--no-small", action="store_true", help="skip the small-N retrain-latency block (BASELINE configs 1-3)")
    ap.add_argument("--no-s4", action="store_true", help="skip the S4 block (BASELINE config 4) of the 1-GPU run")
    ap.add_argument("--s4-maxiter", type=int, default=10)
    ap.add_argument("--s4-budget-s", type=float, default=400.0, help="wall budget of the S4 GP.fit (no new LML evaluation after it)")
    ap.add_argument("--profile-e2e", default=None, help="write a cProfile listing of one end-to-end step to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dump_dir = args.dump_outputs if rank == 0 else None
    n_struct, nrep, seed0, desc = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    config = {"workload": desc, "kernel": "RBF zeta=2 sigma=%g l=%g" % (SIGMA, ELL), "descriptor": "SO3 nmax=3 lmax=4 rcut=5.0 (d=30)",
              "step": "K and dK/dl of the training set (K_ee + K_ef + K_ff, gradient epilogue)",
              "l2": "inputs (packed rows, >300 MB) and outputs (>8 GB) exceed the 126 MB L2; no flush needed"}

    if args.impl == "reference":
        if rank != 0:
            return
        n_cpu = args.cpu_structures or 5
        gf, dt, kind, sample, _ = run_cpu(n_cpu, nrep, seed0, args.steps, max(args.warmup, 0), threads)
        print(json.dumps({"impl": "reference", "metric": "covariance_build_gflops", "value": gf, "unit": "GFLOP/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": threads, "kind": kind, "sample": sample},
                          "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    t_bench0 = time.time()
    block_s = {}

    def mark(name, _last=[time.time()]):
        block_s[name] = round(time.time() - _last[0], 2)
        _last[0] = time.time()

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from gpr_calculator_b200 import _lib, device as gdev, dist as gdist, synthetic as syn
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    lib = _lib.load()

    # ---- synthetic training set, descriptors on the device ------------------------------------------
    labelled = syn.structures(n_struct, nrep, seed0)
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
    y = syn.targets(labelled)
    e_pack = gdev.Pack(E_dev[0], E_dev[1], E_dev[2])
    f_pack = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
    NE, NF = e_pack.n_groups, f_pack.n_groups
    N = NE + 3 * NF
    ele_f, ele_e = F_dev[2].cpu().numpy(), E_dev[1].cpu().numpy()
    p_ff = syn.pair_counts(ele_f, F_dev[3], symmetric=True)          # J >= I blocks only
    p_ee = syn.pair_counts(ele_e, E_dev[2], symmetric=False)
    p_ef = e_pack.pair_count(f_pack)                                  # one pass writes K_ef and K_fe
    flops = flops_of(p_ff, p_ef, p_ee)
    config.update({"N": N, "force_rows": int(F_dev[0].shape[0]), "energy_rows": int(E_dev[0].shape[0]),
                   "pairs_ff_evaluated": p_ff, "parallelism": "row-block x%d" % world,
                   "gather": "none (1 GPU)" if world == 1 else
                   ("fused into the K_fe/K_ff epilogue (NVLink peer stores, gprb_k*_multi)" if gdist.peer_gather_enabled()
                    else "NCCL all-gather (GPRB_NO_PEER=1)")})

    gp = GP(kernel=RBF_mb(para=[SIGMA, ELL], zeta=ZETA), descriptor=des, noise_e=NOISE_E, noise_f=NOISE_F, log_file=None)
    gp.train_x = {"energy": e_pack, "force": f_pack}      # device-resident packs (gdev.packs_of passes Packs through)
    gp.y_train = y

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return gp._build_K(grad=True)

    mark("setup_descriptors_packs")
    # ---- multi-GPU parity, before anything is timed (the driver's GPU test box has one GPU) -----------
    parity_multi = None
    if world > 1:
        pm = sharded_parity(des, nrep, seed0)
        t = torch.tensor([pm["max_rel_K"], pm["max_rel_dK"], pm["lml_rel"], pm["grad_rel"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pm.update({"max_rel_K": float(t[0]), "max_rel_dK": float(t[1]), "lml_rel": float(t[2]), "grad_rel": float(t[3])})
        pm["passed"] = bool(pm["max_rel_K"] <= 1e-12 and pm["max_rel_dK"] <= 1e-12 and pm["lml_rel"] <= 1e-10 and pm["grad_rel"] <= 1e-8)
        pm["what"] = ("row-sharded K / dK/dl (+ LML and gradient) of a %d-row problem against the window-free build on every "
                      "rank, max over ranks" % pm["N"])
        parity_multi = pm
        if not pm["passed"]:
            if rank == 0:
                print(json.dumps({"error": "multi-GPU parity failed", "parity_multi": pm}))
            raise SystemExit(3)

    mark("parity_multi")
    for _ in range(max(args.warmup, 0)):
        out = step()
        del out
    clocks = Clocks(local_rank) if rank == 0 else None
    barrier()
    launches0 = lib.gprb_launch_count()
    _lib.PROFILE = []
    t_wall0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    out = None
    for _ in range(args.steps):
        out = None            # free the previous K and dK/dl before the next build allocates its own
        out = step()
    ev1.record()
    barrier()
    t_wall1 = time.time()
    if dump_dir is not None:
        K_last, dK_last, _ = out
        idx = k_sample_index(NE, N)
        idx_dev = torch.as_tensor(idx, device="cuda")
        dump(dump_dir, "K_sample_index", idx)
        dump(dump_dir, "K_sample", K_last.index_select(0, idx_dev).index_select(1, idx_dev).cpu().numpy())
        if world == 1:        # with several ranks dK/dl holds this rank's rows only, and their windows adapt per build
            dump(dump_dir, "dK_dl_sample", dK_last.index_select(0, idx_dev).index_select(1, idx_dev).cpu().numpy())
        del K_last, dK_last
    del out
    prof, _lib.PROFILE = _lib.PROFILE, None
    launches = lib.gprb_launch_count() - launches0
    ms_step = ev0.elapsed_time(ev1) / args.steps
    kff_ms = [a.elapsed_time(b) for n, a, b, _ in prof if n in ("gprb_kff", "gprb_kff_multi")]
    kff_ms_avg = float(np.mean(kff_ms))
    t = torch.tensor([ms_step, kff_ms_avg], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, kff_ms_max = float(t[0]), float(t[1])
    clk = clocks.summary(t_wall0, t_wall1) if clocks else None

    # ---- roofline of the dominant kernel (K_ff DMMA kernel), per launch on this rank ------------------
    peak = np.zeros(1)
    _lib.call("gprb_fp64_dmma_peak", peak.ctypes.data, gdev.stream())
    if world == 1:
        my_pff = p_ff
    else:
        windows = gdist.row_windows(e_pack.indices, f_pack.indices, world, upper=True)
        (f0, f1) = windows[rank][1]
        rows = np.asarray(f_pack.indices, dtype=np.float64)
        suffix = np.cumsum(rows[::-1])[::-1]
        my_pff = float((rows[f0:f1] * suffix[f0:f1]).sum())
    achieved = 32.0 * D * my_pff / (kff_ms_avg * 1e-3) * 1e-12
    roofline = {"bound": "tensor", "kernel": "cov_mma_kernel<4,8,RBF,grad> (gprb_kff, FP64 DMMA.8x8x4)",
                "achieved": achieved, "peak": float(peak[0]), "unit": "TFLOP/s", "frac": achieved / float(peak[0]),
                "traffic": KFF_DRAM_TRAFFIC.get(args.workload) if world == 1 else None,
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel at this "
                                  "size (profiles/r01_kff_s5_ncu_summary.txt); K and dK/dl written once = 17.05 GB",
                "peak_source": "live DMMA.8x8x4 issue-rate microbenchmark (gprb_fp64_dmma_peak); "
                "MEASURED_PEAKS.json has no fp64 entry; cuBLAS DGEMM 8192^3 on this pool: 35.5 TFLOP/s",
                "kff_ms_per_launch": kff_ms_avg, "algorithmic_flops_per_pair": 32 * D}

    result = {"metric": "covariance_build_gflops", "value": flops / (ms_step * 1e-3) * 1e-9, "unit": "GFLOP/s",
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
              "config": config, "roofline": roofline, "gpu_launches": int(launches), "clocks": clk,
              "k_build_ms": ms_step, "kff_ms_max_over_ranks": kff_ms_max}
    if parity_multi is not None:
        result["parity_multi"] = parity_multi
    if world > 1 and getattr(gp, "_peer", None) is None and gdist.peer_gather_enabled():
        result["config"]["gather"] = "NCCL all-gather (peer mapping unavailable)"

    mark("k_build")
    # ---- end to end: GP.log_marginal_likelihood from pinned host arrays ------------------------------
    if not args.no_e2e:
        E_host, keep1 = syn.to_host(E_dev, pin=True)
        F_host, keep2 = syn.to_host(F_dev, pin=True)
        h2d = sum(a.nbytes for a in E_host[:2]) + sum(a.nbytes for a in F_host[:3])
        gp2 = GP(kernel=RBF_mb(para=[SIGMA, ELL], zeta=ZETA), descriptor=des, noise_e=NOISE_E, noise_f=NOISE_F, log_file=None)
        gp2.train_x = {"energy": E_host, "force": F_host}
        gp2.y_train = y
        theta = np.array([SIGMA, ELL])

        def e2e_step():
            gdev.clear_cache()        # every step re-sends the host arrays and re-packs the rows
            return gp2.log_marginal_likelihood(theta, eval_gradient=True)

        res = None
        for _ in range(min(max(args.warmup, 0), 3)):
            res = e2e_step()
        if args.profile_e2e and rank == 0:
            import cProfile
            import io
            import pstats
            pr = cProfile.Profile()
            pr.enable()
            e2e_step()
            torch.cuda.synchronize()
            pr.disable()
            buf = io.StringIO()
            pstats.Stats(pr, stream=buf).sort_stats("cumulative").print_stats(40)
            with open(args.profile_e2e, "w") as fh:
                fh.write(buf.getvalue())
        elif args.profile_e2e:
            e2e_step()
        barrier()
        _lib.PROFILE = []
        t0 = time.perf_counter()
        step_s = []
        for _ in range(args.steps):
            t_s = time.perf_counter()
            res = e2e_step()
            step_s.append(time.perf_counter() - t_s)      # (the call ends with a host synchronisation: gprb_lml_eval reads its scalars back)
        barrier()
        dt = (time.perf_counter() - t0) / args.steps
        prof, _lib.PROFILE = _lib.PROFILE, None
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t[0])
        parts, host_parts = {}, {}
        for n, a, b, h in prof:
            parts[n] = parts.get(n, 0.0) + a.elapsed_time(b) / args.steps
            host_parts[n] = host_parts.get(n, 0.0) + h * 1e3 / args.steps
        # device -> host reads of a step: 2 doubles per scalar-reducing call, the potrf status word
        # device -> host reads of a step: gprb_lml_eval copies 9 doubles + 2 status words back, once
        d2h = 80 * sum(1 for n, _, _, _ in prof if n == "gprb_lml_eval") / args.steps
        lml, grad = res
        dump(dump_dir, "lml", [lml])
        dump(dump_dir, "lml_grad", grad)
        result["e2e"] = {"value": flops / dt * 1e-9, "unit": "GFLOP/s", "h2d_bytes_per_step": int(h2d),
                         "d2h_bytes_per_step": int(d2h), "ms_per_step": dt * 1e3,
                         "ms_per_step_min_max_on_rank0": [min(step_s) * 1e3, max(step_s) * 1e3],
                         "call": "GP.log_marginal_likelihood(theta, eval_gradient=True) from pinned host packed arrays",
                         "device_ms_by_entry_point": {k: round(v, 3) for k, v in sorted(parts.items())},
                         "host_ms_inside_entry_point": {k: round(v, 3) for k, v in sorted(host_parts.items())},
                         "lml": float(lml), "lml_grad": [float(g) for g in grad]}
        gp2.release_peer()
        del gp2
        gdev.clear_cache()

    mark("e2e")
    # ---- predictions per second against the full training set: BASELINE config 5, "predict 10k structures" ----------
    # 10 000 distinct S5-like test structures (seeds 3000 + k), sharded over the ranks by GP.predict_structures (contiguous
    # blocks, one all-reduce of the results); wall clock from host Atoms to numpy E / F / sigma on every rank.
    if not args.no_predict:
        try:
            gp._alpha_dev = None
            K, _, _ = gp._build_K(grad=False)
            K = gp._own(K)
            gp._alpha_dev = gp._factor(K, NOISE_E, NOISE_F)
            gp._L_dev, gp._Kinv_dev = K, None            # (K is an owned copy)
            gp.fits += 1
            n_test = args.predict_structures
            tests = [a for a, _, _ in syn.structures(n_test, nrep, 3000)]
            # single-structure calls (the reference's route: explicit inverse) on rank-local replicas
            for a in tests[:2]:
                gp.predict_structure(a, stress=False, return_std=True, f_tol=1e-12)
            barrier()
            t0 = time.perf_counter()
            singles = [gp.predict_structure(a, stress=False, return_std=True, f_tol=1e-12) for a in tests[:8]]
            barrier()
            single_ms = (time.perf_counter() - t0) / 8 * 1e3
            pb = args.predict_batch
            gp.predict_structures(tests[:2 * pb * world], return_std=True, f_tol=1e-12, batch=pb)      # warm-up
            barrier()
            _lib.PROFILE = []
            t0 = time.perf_counter()
            res = gp.predict_structures(tests, return_std=True, f_tol=1e-12, batch=pb)
            barrier()
            dt_pred = time.perf_counter() - t0
            prof, _lib.PROFILE = _lib.PROFILE, None
            t = torch.tensor([dt_pred], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_pred = float(t[0])
            predict_parts = {}
            n_batches = max(1, -(-(-(-n_test // world)) // pb))       # ceil(ceil(n_test / world) / batch) batches on the busiest rank
            for n, a, b, h in prof:
                predict_parts[n] = round(predict_parts.get(n, 0.0) + a.elapsed_time(b) / n_batches, 3)
            dE = max(abs(res[k][0] - singles[k][0]) for k in range(8))
            dF = max(float(np.abs(res[k][1] - singles[k][1]).max()) for k in range(8))
            dS = max(max(abs(res[k][3] - singles[k][3]), float(np.abs(res[k][4] - singles[k][4]).max())) for k in range(8))
            assert len(res) == n_test and dE <= 1e-8 and dF <= 1e-8, (dE, dF)
            if dump_dir is not None:
                pick = np.sort(np.random.default_rng(1).choice(n_test, min(n_test, DUMP_STRUCTURES), replace=False))
                for name, k in (("predict_energy", 0), ("predict_forces", 1), ("predict_energy_std", 3), ("predict_forces_std", 4)):
                    dump(dump_dir, name, np.stack([res[i][k] for i in pick]))
                dump(dump_dir, "predict_index", pick)
            # conditioning diagnostic: how far the reference's explicit-inverse variance formula is from the factor route
            from gpr_calculator_b200.batch import rows_from_batch
            E_t, F_t = rows_from_batch(des.calculate_batch(tests[:2], to_host=False), None)
            Xp = {"energy": gdev.energy_pack(E_t), "force": gdev.force_pack(F_t)}
            Ks_p, _ = gp.kernel.k_total_device(Xp, gp.get_train_x(), f_tol=1e-12, grad=False)
            probe = gp.variance_route_probe(Ks_p, gp.kernel.diag_device(Xp))
            result["predict"] = {"value": n_test / dt_pred, "unit": "structures/s", "structures": n_test, "seconds": dt_pred,
                                 "n_train": N, "atoms": len(tests[0]), "single_call_ms": single_ms,
                                 "batch": pb, "device_ms_per_batch_of_32": {k: round(v * 32.0 / pb, 3) for k, v in predict_parts.items()},
                                 "batch_vs_single_max_abs": {"E": dE, "F": dF, "sigma": dS},
                                 "variance_route": "batches: Cholesky factor (trsm); single structures: explicit inverse (the "
                                                   "reference's formula, gaussianprocess.py:904-908)",
                                 "sigma_diff_between_routes_128_rows": probe,
                                 "sharding": "structures in contiguous blocks over %d rank(s), results all-reduced" % world,
                                 "call": "GP.predict_structures(%d Atoms, return_std=True, batch=%d): SO3 + K* + mean + std on device, "
                                         "host Atoms in, numpy E/F/std out on every rank; single_call_ms = one "
                                         "GP.predict_structure(atoms, stress=False, return_std=True)" % (n_test, pb)}
        except Exception as exc:      # the prediction leg must not hide the covariance numbers
            result["predict_error"] = repr(exc)

    mark("predict")
    # ---- descriptor producer: SO3 of the whole training set on the device (host Atoms in, device x / dxdr / seq out) ----
    atoms_list = [a for a, _, _ in labelled]
    des.calculate_batch(atoms_list[:64], to_host=False)
    barrier()
    t0 = time.perf_counter()
    n_seq = 0
    for s0 in range(0, len(atoms_list), 64):
        r = des.calculate_batch(atoms_list[s0:s0 + 64], to_host=False)
        n_seq += int(r["seq"].shape[0])
    barrier()
    dt_so3 = time.perf_counter() - t0
    n_atoms = sum(len(a) for a in atoms_list)
    result["so3"] = {"value": len(atoms_list) / dt_so3, "unit": "structures/s", "atoms_per_structure": n_atoms // len(atoms_list),
                     "seq_rows": n_seq, "output_gb_per_s": 8.0 * (n_atoms * D + n_seq * 3 * D) / dt_so3 * 1e-9,
                     "call": "SO3.calculate_batch(64 structures, to_host=False): neighbour search, radial integrals, power spectrum "
                             "and dx/dr on device; bound by FP64 special functions, not HBM"}

    mark("so3")
    # ---- small-N retrain latency (BASELINE configs 1-3) and S4 (config 4): 1-GPU run only ---------------------------
    if world == 1 and not args.no_small:
        try:
            result["small_n"] = small_n_block(des)
        except Exception as exc:
            result["small_n_error"] = repr(exc)
    mark("small_n")
    if world == 1 and not args.no_s4 and args.workload == "s5":
        try:
            del gp, e_pack, f_pack, E_dev, F_dev
            gdev.clear_cache()
            torch.cuda.empty_cache()
            result["s4"] = s4_block(des, args.s4_maxiter, args.s4_budget_s)
        except Exception as exc:
            result["s4_error"] = repr(exc)

    mark("s4")
    # ---- CPU baseline on the box's host cores (rank 0, N = 1 only) + parity of the CUDA path against it -------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_cpu = args.cpu_structures or 8
        gf, dt, kind, sample, (e_items, f_items, ref) = run_cpu(n_cpu, nrep, seed0, 1, 0, threads)
        result["cpu_baseline"] = {"value": gf, "unit": "GFLOP/s", "cores": threads, "kind": kind, "sample": sample,
                                  "seconds": dt}
        if SO3_CPU_SECONDS:
            result["so3"]["cpu_port_structures_per_s"] = 1.0 / float(np.mean(SO3_CPU_SECONDS))
            result["so3"]["cpu_port"] = "oracle/so3.py (numpy restatement of SO3.calculate), 1 core, same structures"
        result["parity"] = parity_vs_reference(e_items, f_items, ref[0], ref[1], [syn.cu_fcc(nrep, seed0 + k)[0] for k in range(n_cpu)])
        if not result["parity"]["passed"]:
            print(json.dumps({"error": "parity against the reference failed", "parity": result["parity"]}))
            raise SystemExit(4)
    mark("cpu_baseline_parity")
    result["bench_seconds"] = dict(block_s, total=round(time.time() - t_bench0, 2))
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        gp.release_peer()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
