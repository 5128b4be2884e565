"""Worker of tests/test_gpu_virial.py::test_sharded_stress_predictions_match_unsharded (run under torchrun, one rank per
GPU): GP.predict_structures(stress=True, return_std=True) sharded over the ranks against every rank predicting the whole
list (shard=False)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rank, world = dist.get_rank(), dist.get_world_size()
    from gpr_calculator_b200 import device as gdev, synthetic as syn
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb

    n_struct = 12
    labelled = syn.structures(n_struct, 2, 2000)
    des = SO3(nmax=3, lmax=4, rcut=5.0, stress=True)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
    y = syn.targets(labelled)
    gp = GP(kernel=RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    gp.train_x = {"energy": gdev.Pack(E_dev[0], E_dev[1], E_dev[2]),
                  "force": gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])}
    gp.train_y = {"energy": list(y[:n_struct, 0]), "force": y[n_struct:, 0].reshape(-1, 3)}
    gp.update_y_train()
    gp.N_energy, gp.N_forces = n_struct, n_struct * 32
    gp.fit(opt=False, show=False)
    tests_ = [a for a, _, _ in syn.structures(2 * world + 3, 2, 3000)]
    sharded = gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=4, stress=True)
    local = gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=4, shard=False, stress=True)
    gp.release_peer()
    err = 0.0
    for a, b in zip(sharded, local):
        err = max(err, abs(a[0] - b[0]), abs(a[3] - b[3]),
                  *(float(np.abs(np.asarray(u) - np.asarray(v)).max()) for u, v in ((a[1], b[1]), (a[2], b[2]), (a[4], b[4]),
                                                                                    (a[5], b[5]))))
    ok = len(sharded) == len(tests_) and all(len(t) == 6 for t in sharded) and err <= 1e-9
    print("[rank %d/%d] sharded stress predictions max |diff| vs replicated %.2e" % (rank, world, err), flush=True)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
