"""Row-block sharding of the covariance matrix over GPUs (one process per GPU, NCCL via torch.distributed).

Replaces the reference's mpi4py pattern — every rank computes a row slab, rank 0 gathers pickles,
vstacks and broadcasts (RBF_mb.py:471-521, gaussianprocess.py:246-247,305-306) — with:
  * contiguous row blocks of training groups balanced by cost (rows of the group),
  * one in-place all-gather of the slabs into the full K on every GPU,
  * dK/dtheta never gathered: each rank traces its own rows, scalars are all-reduced.
With the gloo backend (CPU tensors) the same partition / gather logic is exercised in the tests.

On one NVLink / NVSwitch node the gather is fused into the covariance kernels instead (PeerMatrix): every
rank's copy of K is mapped into every other process, the kernel epilogue stores each finished value into all
copies, and two stream-ordered rank barriers replace the all-gather.
"""
import ctypes
import os
import warnings
import weakref

import numpy as np
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def split_groups(costs, parts, speed=None):
    """Contiguous partition of len(costs) groups into `parts` blocks with balanced total cost
    (block p gets a share proportional to speed[p] when given).

    Returns `parts + 1` boundaries b with b[0] = 0 and b[-1] = len(costs)."""
    costs = np.asarray(costs, dtype=np.float64)
    n = len(costs)
    if n == 0:
        return [0] * (parts + 1)
    cum = np.concatenate(([0.0], np.cumsum(costs)))
    total = cum[-1]
    share = np.ones(parts) if speed is None else np.asarray(speed, dtype=np.float64)
    share = np.cumsum(share) / share.sum()
    bounds = [0]
    for p in range(1, parts):
        target = total * share[p - 1]
        j = int(np.searchsorted(cum, target, side="left"))
        if j > 0 and abs(cum[j - 1] - target) <= abs(cum[min(j, n)] - target):
            j -= 1
        j = min(max(j, bounds[-1]), n)
        bounds.append(j)
    bounds.append(n)
    return bounds


def row_windows(e_rows, f_rows, parts, upper=False, speed=None):
    """Per-rank windows ((e0,e1),(f0,f1)) over energy groups and force groups.

    Energy and force groups are partitioned independently so that every rank gets an equal share
    of both block rows (the force block dominates: cost ~ rows of the centre).  upper=True balances
    the trapezoids of an upper-triangle build (GPRB_FF_UPPER): force group I costs
    n_I * sum_{J >= I} n_J.  speed[r] (relative measured throughput of rank r, see GP._build_K) scales
    the share of the force rows rank r receives."""
    eb = split_groups(e_rows, parts)
    f = np.asarray(f_rows, dtype=np.float64)
    if upper and len(f):
        f = f * np.cumsum(f[::-1])[::-1]
    fb = split_groups(f, parts, speed=speed)
    return [((eb[r], eb[r + 1]), (fb[r], fb[r + 1])) for r in range(parts)]


def window_row_ranges(windows, NE):
    """Row ranges in the assembled matrix covered by each window: list of [(lo,hi) energy, (lo,hi) force]."""
    return [((e0, e1), (NE + 3 * f0, NE + 3 * f1)) for (e0, e1), (f0, f1) in windows]


def gather_rows(K_local, windows, NE, N, group=None):
    """All-gather row slabs into the full [N, N_cols] matrix on every rank.

    K_local holds this rank's rows: first its energy rows, then its force rows."""
    rank, size = world()
    n_cols = K_local.shape[1]
    if size == 1:
        return K_local
    K = torch.empty((N, n_cols), dtype=K_local.dtype, device=K_local.device)
    (e0, e1), (f0, f1) = windows[rank]
    K[e0:e1] = K_local[:e1 - e0]
    K[NE + 3 * f0:NE + 3 * f1] = K_local[e1 - e0:]
    gather_rows_inplace(K, windows, NE, group=group)
    return K


def gather_rows_inplace(K, windows, NE, group=None):
    """In-place all-gather: every rank has written its own energy and force row slabs of the full
    matrix K; on return every rank holds all rows.  The slabs are contiguous row ranges of the
    row-major matrix, so each is sent from and received into K itself (no staging copies); uneven
    slab sizes are handled by the backend (NCCL: grouped broadcasts)."""
    rank, size = world()
    if size == 1:
        return K
    for slabs in ([K[e0:e1] for (e0, e1), _ in windows], [K[NE + 3 * f0:NE + 3 * f1] for _, (f0, f1) in windows]):
        if all(s.numel() == 0 for s in slabs):
            continue
        n0 = slabs[0].numel()
        lo = slabs[0].data_ptr()
        if n0 > 0 and all(s.numel() == n0 and s.data_ptr() == lo + r * n0 * K.element_size() for r, s in enumerate(slabs)):
            # equal slabs tiling one contiguous range: a single all-gather straight into K
            whole = K.view(-1)[(lo - K.data_ptr()) // K.element_size():][:size * n0]
            dist.all_gather_into_tensor(whole, slabs[rank].reshape(-1).clone(), group=group)
            continue
        # uneven slabs (cost-balanced windows): one broadcast per owner, each received in place
        for r, s in enumerate(slabs):
            if s.numel():
                dist.broadcast(s, src=r if group is None else dist.get_global_rank(group, r), group=group)
    return K


def all_gather_floats(value, device="cpu", group=None):
    """One python float per rank -> list of all ranks' values."""
    rank, size = world()
    if size == 1:
        return [float(value)]
    t = torch.zeros(size, dtype=torch.float64, device=device)
    t[rank] = float(value)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return [float(v) for v in t.cpu()]


def broadcast_floats(values, src=0, device="cpu", group=None):
    """Every rank returns rank `src`'s list of python floats."""
    rank, size = world()
    if size == 1:
        return [float(v) for v in values]
    t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=device)
    dist.broadcast(t, src=src if group is None else dist.get_global_rank(group, src), group=group)
    return [float(v) for v in t.cpu()]


def all_reduce_sum(values, device="cpu", group=None):
    """Sum a small list of python floats over ranks."""
    rank, size = world()
    if size == 1:
        return list(values)
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return [float(v) for v in t.cpu()]


def all_to_all_rows(out, inp, recv_rows, send_rows, group=None):
    """Exchange contiguous row blocks of two row-major matrices with the same row length: this rank sends send_rows[d]
    consecutive rows of `inp` to rank d (in rank order) and receives recv_rows[s] rows from rank s into `out`
    (in rank order).  Point-to-point sends / receives in one batch (NCCL: one grouped launch over NVLink; gloo in the tests);
    the rank's own block is a local copy."""
    rank, size = world()
    assert out.shape[1] == inp.shape[1] and sum(send_rows) == inp.shape[0] and sum(recv_rows) == out.shape[0]
    so = np.concatenate(([0], np.cumsum(send_rows))).astype(int)
    ro = np.concatenate(([0], np.cumsum(recv_rows))).astype(int)
    ops = []
    for p in range(size):
        peer = p if group is None else dist.get_global_rank(group, p)
        if p == rank:
            if send_rows[p]:
                out[ro[p]:ro[p + 1]] = inp[so[p]:so[p + 1]]
            continue
        if send_rows[p]:
            ops.append(dist.P2POp(dist.isend, inp[so[p]:so[p + 1]], peer, group=group))
        if recv_rows[p]:
            ops.append(dist.P2POp(dist.irecv, out[ro[p]:ro[p + 1]], peer, group=group))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    return out


def distributed_cholesky(K, nb=1024, group=None, panel_fn=None, trailing_fn=None):
    """In-place Cholesky factorisation K = L L^T of a symmetric matrix that EVERY rank holds in full (row-major [N, N] CUDA
    tensor; on return the row-major lower triangle of every rank's copy holds L, the strict upper triangle is undefined).

    Right-looking blocked algorithm, block column k of the lower triangle owned by rank k mod G: the owner factors the
    diagonal block and solves for the rows below (gprb_chol_panel: cuSOLVER potrf + cuBLAS trsm), the finished panel is
    broadcast over NVLink (NCCL) into every copy, and every rank applies the rank-nb update to the block columns it owns
    (gprb_chol_trailing: one cuBLAS gemm per column).  All steps are stream ordered; one host synchronisation at the end
    reads the status.  Replaces the factorisation the reference repeats on every MPI rank (gaussianprocess.py:174): with G
    ranks the N^3 / 3 flops are split G ways (S5 on 8 B200: 0.36 s replicated -> see DESIGN.md).
    Returns potrf's info (0 = positive definite), identical on every rank.
    panel_fn(K, k0, nbk, info) / trailing_fn(K, k0, nbk, j0, nbj): the two arithmetic steps; default = the library entry points
    (the gloo test of the ownership / broadcast logic passes numpy stand-ins)."""
    rank, size = world()
    N = int(K.shape[0])
    info = torch.zeros(1, dtype=torch.int32, device=K.device)
    if panel_fn is None:
        from . import _lib
        from .device import ptr, stream
        ld, st = int(K.stride(0)), stream()

        def panel_fn(K, k0, nbk, info):
            _lib.call("gprb_chol_panel", ptr(K), ld, N, k0, nbk, ptr(info), st)

        def trailing_fn(K, k0, nbk, j0, nbj):
            _lib.call("gprb_chol_trailing", ptr(K), ld, N, k0, nbk, j0, nbj, st)
    nblk = -(-N // nb)
    for k in range(nblk):
        k0, nbk = k * nb, min(nb, N - k * nb)
        owner = k % size
        if owner == rank:
            panel_fn(K, k0, nbk, info)
        if size > 1:
            # the panel (rows k0..N of block column k) travels as one contiguous buffer
            panel = K[k0:, k0:k0 + nbk]
            buf = panel.contiguous() if owner == rank else torch.empty((N - k0, nbk), dtype=K.dtype, device=K.device)
            dist.broadcast(buf, src=owner if group is None else dist.get_global_rank(group, owner), group=group)
            if owner != rank:
                panel.copy_(buf)
        for j in range(k + 1, nblk):
            if j % size == rank:
                trailing_fn(K, k0, nbk, j * nb, min(nb, N - j * nb))
    if size > 1:
        dist.all_reduce(info, op=dist.ReduceOp.MAX, group=group)
    return int(info.item())


def all_reduce_array(values, device="cpu", group=None):
    """Element-wise sum of a 1-D float64 numpy array over ranks (sharded prediction: every rank fills its own slots of a
    zero array, so the sum is an exact gather)."""
    rank, size = world()
    values = np.ascontiguousarray(values, dtype=np.float64)
    if size == 1:
        return values
    t = torch.from_numpy(values).to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def gather_predictions(mine, n_atoms, first, return_std, device="cpu", group=None, stress=False):
    """Combine per-rank prediction results into the full list on every rank.

    mine: this rank's results for the structures [first, first + len(mine)) of a list whose structures have
    n_atoms[k] atoms: tuples (E, F [n, 3], None) or (E, F, None, E_std, F_std [n, 3]).  Flat layout per structure:
    E, F (3 n) [, E_std, F_std (3 n)]; every rank fills its own slots of a zero buffer, one all-reduce.
    stress=True: tuples (E, F, S [6]) or (E, F, S, E_std, F_std, S_std [6]); S follows F and S_std follows F_std."""
    width = 2 if return_std else 1
    ns = 6 if stress else 0
    sizes = np.array([(1 + 3 * n + ns) * width for n in n_atoms], dtype=np.int64)
    offs = np.concatenate(([0], np.cumsum(sizes)))
    flat = np.zeros(int(offs[-1]))
    for k, res in enumerate(mine):
        o, n3 = int(offs[first + k]), 3 * n_atoms[first + k]
        h = 1 + n3 + ns                      # start of the standard deviations
        flat[o] = res[0]
        flat[o + 1:o + 1 + n3] = np.asarray(res[1]).reshape(-1)
        if stress:
            flat[o + 1 + n3:o + h] = res[2]
        if return_std:
            flat[o + h] = res[3]
            flat[o + h + 1:o + h + 1 + n3] = np.asarray(res[4]).reshape(-1)
            if stress:
                flat[o + h + 1 + n3:o + 2 * h] = res[5]
    flat = all_reduce_array(flat, device=device, group=group)
    out = []
    for k, n in enumerate(n_atoms):
        o, n3 = int(offs[k]), 3 * n
        h = 1 + n3 + ns
        F = flat[o + 1:o + 1 + n3].reshape(-1, 3).copy()
        S = flat[o + 1 + n3:o + h].copy() if stress else None
        if return_std:
            res = (float(flat[o]), F, S, float(flat[o + h]), flat[o + h + 1:o + h + 1 + n3].reshape(-1, 3).copy())
            out.append(res + ((flat[o + h + 1 + n3:o + 2 * h].copy(),) if stress else ()))
        else:
            out.append((float(flat[o]), F, S))
    return out


# ------------------------------------------------------------------------------------------------
# fused gather: K of every rank mapped into every process (CUDA IPC over NVLink peer access)
# ------------------------------------------------------------------------------------------------
class _RawDeviceArray:
    """Device memory owned by libgpr_b200 (gprb_peer_alloc) exposed through __cuda_array_interface__ so
    that torch can view it (torch stays the owner of streams and the tensor algebra around it)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def slab_pointers(bases, row0, col0, ld, itemsize=8):
    """Pointer to element (row0, col0) of the same row-major matrix at each base address."""
    return [int(b) + (int(row0) * int(ld) + int(col0)) * itemsize for b in bases]


class PeerMatrix:
    """An [N, N] float64 matrix per rank, every rank's copy mapped into every other process.

    `tensor` is this rank's copy; `ptrs[r]` is the device address of rank r's copy as seen from this
    process (ptrs[rank] is the local one).  Writers store into all copies (gprb_kff_multi /
    gprb_kfe_multi); `barrier()` is a stream-ordered rank barrier (a one-element all-reduce on the current
    stream): work enqueued after it on any rank starts after the work enqueued before it on every rank.
    Collective: every rank of the group must construct / close it together."""

    def __init__(self, N, group=None):
        from . import _lib
        rank, size = world()
        self.N, self.rank, self.size, self.group = int(N), rank, size, group
        self.ptrs, self._opened, self._local, self.tensor = [], [], ctypes.c_void_p(0), None
        nbytes = self.N * self.N * 8

        def agreed(ok):
            """Collective: True only if every rank succeeded so far (every rank takes part in every collective of the
            constructor, whatever happened locally, so a local failure can never leave the others waiting)."""
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            return int(flag.item()) == 1

        handle = ctypes.create_string_buffer(64)
        err = ""
        try:       # a second N x N buffer: may fail on a full device, on this rank only
            _lib.call("gprb_peer_alloc", ctypes.byref(self._local), ctypes.c_ulonglong(nbytes))
            _lib.call("gprb_peer_export", self._local, handle)
            ok = True
        except _lib.GprB200Error as exc:
            ok, err = False, str(exc)
        if not agreed(ok):
            self._release()
            raise RuntimeError("peer allocation of K failed on at least one rank %s" % err)
        mine = torch.frombuffer(bytearray(handle.raw), dtype=torch.uint8).cuda()
        every = torch.empty(size * 64, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(every, mine, group=group)
        every = bytes(every.cpu().numpy().tobytes())
        ptrs = []
        for r in range(size):
            if r == rank:
                ptrs.append(int(self._local.value))
                continue
            q = ctypes.c_void_p(0)
            try:
                _lib.call("gprb_peer_open", every[64 * r:64 * (r + 1)], ctypes.byref(q))
                self._opened.append(q)
                ptrs.append(int(q.value))
            except _lib.GprB200Error as exc:      # no peer access to that GPU (not one NVLink node?)
                ok, err = False, str(exc)
                ptrs.append(0)
        if not agreed(ok):
            self._release()
            raise RuntimeError("peer mapping of K failed on at least one rank %s" % err)
        self.ptrs = ptrs
        self.tensor = torch.as_tensor(_RawDeviceArray(self._local.value, (self.N, self.N)), device="cuda")
        self._token = torch.zeros(1, dtype=torch.int32, device="cuda")
        # best effort when a GP is dropped without release_peer(): unmap the peers and free the local buffer (not collective;
        # a peer that still stores into this copy is a caller error, as with close())
        self._finalizer = weakref.finalize(self, PeerMatrix._free, self._opened, self._local)

    @staticmethod
    def _free(opened, local):
        try:
            from . import _lib
            lib = _lib.load()
            for q in opened:
                lib.gprb_peer_close(q)
            del opened[:]
            if local:
                lib.gprb_peer_free(local)
                local.value = None
        except Exception:
            pass

    def barrier(self):
        dist.all_reduce(self._token, group=self.group)

    def _release(self):
        PeerMatrix._free(self._opened, self._local)
        self.ptrs = []

    def close(self):
        """Collective: nobody may still be writing into anybody's copy."""
        if self._local:
            self.barrier()
            torch.cuda.synchronize()
            self.tensor = None
            from . import _lib
            for q in self._opened:          # unmap the peers' copies first, then everyone frees its own
                _lib.load().gprb_peer_close(q)
            del self._opened[:]
            self.barrier()
            torch.cuda.synchronize()
            self._release()


def peer_gather_enabled():
    """The fused gather is used for multi-GPU builds unless GPRB_NO_PEER=1 (then: NCCL all-gather)."""
    return os.environ.get("GPRB_NO_PEER", "0") in ("", "0")


def make_peer_matrix(N, group=None):
    """PeerMatrix or None (with a warning) when the ranks cannot map each other's memory."""
    try:
        return PeerMatrix(N, group=group)
    except RuntimeError as exc:      # same outcome on every rank (every step's success flag is all-reduced)
        warnings.warn("fused peer gather unavailable, using the NCCL all-gather: %s" % exc)
        return None
