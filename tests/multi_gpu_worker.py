"""Worker of tests/test_gpu_multi.py (run under torchrun, one rank per GPU): the row-sharded covariance build
with the gather fused into the kernels (NVLink peer stores) against the NCCL all-gather build and the
single-GPU build of the same training set, then LML + gradient through the sharded paths against the reference's
algebra evaluated on the host (oracle.gp.lml_from_matrices) on the unsharded K and dK/dl."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    n_struct = int(sys.argv[1]) if len(sys.argv) > 1 else 24
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rank, world = dist.get_rank(), dist.get_world_size()
    from gpr_calculator_b200 import device as gdev, synthetic as syn
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from oracle import gp as ogp

    labelled = syn.structures(n_struct, 2, 2000)
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
    y = syn.targets(labelled)
    e_pack = gdev.Pack(E_dev[0], E_dev[1], E_dev[2])
    f_pack = gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
    theta = np.array([1.0, 0.1])

    def make_gp():
        gp = GP(kernel=RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
        gp.train_x = {"energy": e_pack, "force": f_pack}
        gp.train_y = {"energy": list(y[:n_struct, 0]), "force": y[n_struct:, 0].reshape(-1, 3)}
        gp.update_y_train()
        gp.N_energy, gp.N_forces = e_pack.n_groups, f_pack.n_groups
        return gp

    # single-GPU build of the whole matrix on every rank (symmetric mode, no sharding)
    gp0 = make_gp()
    K1, dK1 = gp0.kernel.k_total_device(gp0.train_x, None, f_tol=1e-10, grad=True)
    scale = float(K1.abs().max())
    NE = e_pack.n_groups
    K1h = K1.cpu().numpy()
    lml_h, g_h = ogp.lml_from_matrices(K1h, np.dstack((2 * K1h / theta[0], dK1.cpu().numpy())), y, NE, 0.002, 0.1)

    results = {}
    for mode in ("peer", "nccl", "distchol"):
        os.environ["GPRB_NO_PEER"] = "1" if mode == "nccl" else "0"
        # "distchol": the factorisation shared by the ranks (dist.distributed_cholesky, panels of 256 rows) instead of repeated on each
        GP.DIST_CHOLESKY_MIN_N = 512 if mode == "distchol" else 10 ** 9
        os.environ["GPRB_DIST_CHOLESKY_NB"] = "256"
        gp = make_gp()
        for it in range(3):            # repeated builds re-use (and re-zero) the peer-mapped matrix
            K, dK, ranges = gp._build_K(grad=True)
            K = K.clone()
        if mode != "nccl":
            assert gp._peer is not None, "peer mapping failed: the fused gather was not exercised"
        else:
            assert getattr(gp, "_peer", None) is None
        err = float((K - K1).abs().max()) / scale
        # dK rows held by this rank (energy rows: K_ee part only; force rows: K_fe and the J >= I blocks)
        off, derr = 0, 0.0
        for (r0, r1) in ranges:
            rows = dK[off:off + (r1 - r0)]
            ref = dK1[r0:r1]
            if r1 <= NE:
                derr = max(derr, float((rows[:, :NE] - ref[:, :NE]).abs().max()) if r1 > r0 else 0.0)
            else:
                mask = torch.ones_like(ref, dtype=torch.bool)
                cols = torch.arange(ref.shape[1], device="cuda")
                rr = torch.arange(r0, r1, device="cuda")
                blk_r = (rr - NE) // 3
                blk_c = (cols - NE) // 3
                mask = (cols[None, :] < NE) | (blk_c[None, :] >= blk_r[:, None])
                derr = max(derr, float(((rows - ref).abs() * mask).max()))
            off += r1 - r0
        derr /= float(dK1.abs().max())
        lml, grad = gp.log_marginal_likelihood(theta, eval_gradient=True)
        results[mode] = (K, err, derr, lml, grad)
        gp.release_peer()
    Kp, Kn = results["peer"][0], results["nccl"][0]
    # equal up to the summation order of row groups that straddle two CTAs: the throughput-adaptive row windows
    # (GP._build_K) may cut the rows differently in the two runs
    bitwise = bool(torch.equal(Kp, Kn))
    same = float((Kp - Kn).abs().max()) <= 1e-13 * scale
    lml_p, g_p = results["peer"][3], results["peer"][4]
    lml_n, g_n = results["nccl"][3], results["nccl"][4]
    lml_d, g_d = results["distchol"][3], results["distchol"][4]
    GP.DIST_CHOLESKY_MIN_N = 512          # the fit / prediction checks below run on the shared factorisation too
    # Dot kernel: the d/dsigma0 term of the sharded gradient (E-E constant of dot_kernel.py:58) against the host
    from gpr_calculator_b200.kernels import Dot_mb
    gd_ = GP(kernel=Dot_mb(para=[2.0, 1.5], zeta=3), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    gd_.train_x = {"energy": e_pack, "force": f_pack}
    gd_.y_train = y
    dot = gd_.log_marginal_likelihood(np.array([2.0, 1.5]), eval_gradient=True)
    gd_.release_peer()
    Kd = gd_.kernel.k_total_device(gd_.train_x, None, grad=True)[0].cpu().numpy()
    Cs0 = np.zeros_like(Kd)
    Cs0[:NE, :NE] = 0.8 * 2 * 2.0 ** 2 * 1.5
    dot_h = ogp.lml_from_matrices(Kd, np.dstack((2 * Kd / 2.0, Cs0)), y, NE, 0.002, 0.1)
    dot_ok = abs(dot[0] - dot_h[0]) <= 1e-9 * abs(dot_h[0]) and np.allclose(dot[1], dot_h[1], rtol=1e-7, atol=1e-7)
    # sharded prediction (structures split over the ranks, results all-reduced) against every rank predicting everything,
    # and a full fit with the optimiser values broadcast from rank 0: identical hyper-parameters on every rank
    os.environ["GPRB_NO_PEER"] = "0"
    gpp = make_gp()
    gpp.fit(opt=True, show=False, maxiter=3)
    theta_fit = torch.tensor(gpp.kernel.parameters(), dtype=torch.float64, device="cuda")
    lo, hi = theta_fit.clone(), theta_fit.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    same_theta = bool(torch.equal(lo, hi))
    tests_ = [a for a, _, _ in syn.structures(2 * world + 3, 2, 3000)]
    sharded = gpp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=4)
    local = gpp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=4, shard=False)
    pred_err = max(max(abs(a[0] - b[0]), float(np.abs(a[1] - b[1]).max()), abs(a[3] - b[3]), float(np.abs(a[4] - b[4]).max()))
                   for a, b in zip(sharded, local))
    gpp.release_peer()
    pred_ok = len(sharded) == len(tests_) and pred_err <= 1e-9 and same_theta
    if rank == 0:
        print("sharded prediction max |diff| vs replicated %.2e, fitted theta identical on all ranks: %s (%s)"
              % (pred_err, same_theta, gpp.kernel.parameters()), flush=True)
    ok = (pred_ok and results["peer"][1] <= 1e-12 and results["nccl"][1] <= 1e-12 and results["peer"][2] <= 1e-12 and same
          and abs(lml_p - lml_n) <= 1e-9 * abs(lml_n) and np.allclose(g_p, g_n, rtol=1e-9, atol=1e-9)
          and abs(lml_p - lml_h) <= 1e-9 * abs(lml_h) and np.allclose(g_p, g_h, rtol=1e-7, atol=1e-7) and dot_ok
          and abs(lml_p - lml_d) <= 1e-10 * abs(lml_p) and np.allclose(g_p, g_d, rtol=1e-8, atol=1e-8))
    if rank == 0:
        print("gradient rows %s | host %s | shared Cholesky %s (lml %.12g vs %.12g, host %.12g); Dot rows %s | host %s"
              % (g_p, g_h, g_d, lml_d, lml_p, lml_h, dot, dot_h), flush=True)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    print("[rank %d/%d] N=%d K err peer %.2e nccl %.2e dK err %.2e bitwise(peer,nccl)=%s lml %.9f / %.9f grad %s / %s"
          % (rank, world, K1.shape[0], results["peer"][1], results["nccl"][1], results["peer"][2], bitwise, lml_p, lml_n,
             g_p, g_n), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
