"""CPU, world_size 2, gloo: gather_predictions with the total-stress slots (GP.predict_structures(stress=True)), and the
flat layout without them unchanged."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, size, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    from gpr_calculator_b200 import dist as gd
    n_atoms = [3, 1, 4, 1, 5, 9, 2]
    truth = [(float(k), np.full((n, 3), k + 0.5), np.arange(6) + 10.0 * k, 10.0 + k, np.full((n, 3), k + 0.25),
              np.arange(6) * 0.5 + k) for k, n in enumerate(n_atoms)]
    b = gd.split_groups(n_atoms, size)
    flats = []
    reduce = gd.all_reduce_array

    def spy(values, **kw):
        out = reduce(values, **kw)
        flats.append(out.copy())
        return out

    gd.all_reduce_array = spy
    ok = True
    for std in (False, True):
        mine = [(t[0], t[1], t[2]) + ((t[3], t[4], t[5]) if std else ()) for t in truth[b[rank]:b[rank + 1]]]
        got = gd.gather_predictions(mine, n_atoms, b[rank], std, stress=True)
        for t, g in zip(truth, got):
            ok = ok and len(g) == (6 if std else 3) and g[0] == t[0] and np.array_equal(g[1], t[1])
            ok = ok and np.array_equal(g[2], t[2])
            if std:
                ok = ok and g[3] == t[3] and np.array_equal(g[4], t[4]) and np.array_equal(g[5], t[5])
        # without stress: the layout of earlier releases, E, F (3 n) [, E_std, F_std (3 n)] per structure
        mine = [(t[0], t[1], None) + ((t[3], t[4]) if std else ()) for t in truth[b[rank]:b[rank + 1]]]
        got = gd.gather_predictions(mine, n_atoms, b[rank], std)
        legacy = np.concatenate([np.concatenate(([t[0]], t[1].ravel()) + (([t[3]], t[4].ravel()) if std else ()))
                                 for t in truth])
        ok = ok and np.array_equal(flats[-1], legacy)
        for t, g in zip(truth, got):
            ok = ok and len(g) == (5 if std else 3) and g[2] is None and g[0] == t[0] and np.array_equal(g[1], t[1])
    q.put((rank, ok))
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_gather_predictions_with_stress_two_ranks():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=100) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for rank, ok in res:
        assert ok, "rank %d gathered wrong predictions" % rank
