"""Gaussian-process regressor with the covariance hot path on the B200.

Drop-in for ``gpr_calc.gaussianprocess.GP`` (gaussianprocess.py:22-1161): same constructor, public
methods, training-set containers, printed ``Loss:`` lines and guard behaviour.  What changed is
where the arithmetic runs:

* ``log_marginal_likelihood`` / ``fit`` (gaussianprocess.py:133-202, 222-317): K and dK/dl are
  built on device by the kernel object, the noise is added, Cholesky / alpha come from cuSOLVER
  (potrf / potrs), the rows of K^-1 the gradient needs from triangular solves, and the gradient is
  the trace kernel of libgpr_b200 — K never visits the host.  L-BFGS-B stays scipy on the host, as in the reference (:215-219).
* ``predict`` / ``predict_structure`` (:319-379, 834-918): K* on device, mean and variance with
  the explicit K^-1 the reference uses (:128-131, 904-908), negative variances clipped to 0.
* multi-GPU: with torch.distributed initialised (one process per GPU), each rank builds a row
  block of K / dK, K is all-gathered, the gradient trace is all-reduced (dist.py).  This replaces
  the mpi4py gather/bcast and the redundant allreduce of :246-247.

Persistence (:632-821): the json model file plus an ASE sqlite database of the labelled structures,
read and written by gpr_calculator_b200.asedb (ASE's file layout, no ASE needed); GP.load recomputes
the descriptors in batches on the device.
"""
import ctypes
import json
import logging
import os
from copy import deepcopy

import numpy as np
import torch
from scipy.optimize import minimize

from . import _lib
from . import dist as gdist
from .device import F64, c_vp, packs_of, ptr, require_cuda, stream
from .kernels.Dot_mb import Dot_mb
from .kernels.RBF_mb import RBF_mb
from .utilities import (atomic_numbers, convert_train_data, force_rows, list_to_tuple, metric_values, new_pt,
                        tuple_to_list)


def _zero_build_targets(K, NE, chunks=16):
    """Zero what a row-sharded upper-triangle build accumulates into: the K_fe columns and the part of the
    force-force block on and right of the diagonal (in `chunks` row bands; everything else is overwritten by the
    mirror / transpose / K_ee copies that follow)."""
    N = K.shape[0]
    if N <= NE:
        return
    if NE:
        K[NE:, :NE].zero_()
    per = 3 * max(1, -(-((N - NE) // 3) // chunks))
    for r in range(NE, N, per):
        K[r:r + per, r:].zero_()


def _row_pieces(r_ranges, NE, N, parts=16, min_rows=512):
    """Blocks of rows for the inverse-rows likelihood gradient: the row ranges a rank holds (their rows of dK
    stored one range after the other) cut at the energy / force boundary and, for force rows, into blocks of
    about N / parts rows (>= min_rows).  Returns [(r0, r1, first row of the block inside dK)]."""
    blk = max(min_rows, -(-N // parts))
    pieces = []
    off = 0
    for (r0, r1) in r_ranges:
        cuts = [r0] + ([NE] if r0 < NE < r1 else [])
        a = cuts[-1]
        while a < r1 and a >= NE:     # force rows
            a = min(a + blk, r1)
            cuts.append(a)
        if cuts[-1] != r1:
            cuts.append(r1)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                pieces.append((a, b, off + (a - r0)))
        off += r1 - r0
    return pieces


def _lazy_SO3():
    from .SO3 import SO3
    return SO3


class GP():
    """
    Gaussian Process Regressor class to fit the interatomic potential from reference energy/forces.

    Main APIs: fit(), predict_structure(struc), add_structure((struc, energy, forces)), sparsify()

    Args:
        kernel (callable): compute the covariance matrix
        descriptor (callable): compute the structure to descriptor
        base_potential (callable): compute the base potential before GPR
        f_coef (float): the coefficient of force noise relative to energy
        noise_e (float or list): energy noise, or [init, lower, upper] to optimise it
    """

    def __init__(self, kernel, descriptor,
                 base_potential=None,
                 noise_e=0.005,
                 noise_f=0.1,
                 f_coef=10,
                 log_file="gpr.log"):

        self.log_file = log_file
        self.logging = logging.getLogger("gpr_calculator_b200.%x" % id(self))
        self.logging.setLevel(logging.INFO)
        self.logging.propagate = False
        if log_file is not None and not self.logging.handlers:
            try:
                h = logging.FileHandler(log_file)
                h.setFormatter(logging.Formatter('%(asctime)s| %(message)s'))
                self.logging.addHandler(h)
            except OSError:
                self.logging.addHandler(logging.NullHandler())

        self.rank, self.size = gdist.world()
        if type(noise_e) is not list:
            self.noise_e = noise_e
            self.noise_f = noise_f
            self.noise_bounds = None
        else:
            self.noise_e = noise_e[0]
            self.noise_f = noise_f[0]
            self.noise_bounds = noise_e[1:]
        self.f_coef = f_coef
        self.error = None

        self.descriptor = descriptor
        self.kernel = kernel
        self.base_potential = base_potential

        self.x = None
        self.train_x = None
        self.train_y = None
        self.train_db = None
        self._alpha_dev = None
        self._L_dev = None
        self._Kinv_dev = None
        self.N_energy = 0
        self.N_forces = 0
        self.N_energy_queue = 0
        self.N_forces_queue = 0
        self.N_queue = 0

        self.fits = 0
        self.use_base = 0
        self.use_surrogate = 0
        # device timers of the last fit (ms): covariance builds vs library factorisations
        self.timings = {}

        if self.rank == 0:
            self.logging.info(self)

    # -- numpy views of the device-resident factors (reference attributes L_, alpha_, _K_inv) ----
    @property
    def alpha_(self):
        return None if self._alpha_dev is None else self._alpha_dev.cpu().numpy().reshape(-1, 1)

    @alpha_.setter
    def alpha_(self, v):
        self._alpha_dev = None if v is None else torch.as_tensor(np.asarray(v, dtype=np.float64).ravel(), device="cuda")

    @property
    def L_(self):
        if self._L_dev is None:
            return None
        return np.tril(self._L_dev.cpu().numpy())       # the factor lives in the row-major lower triangle

    @L_.setter
    def L_(self, v):
        self._L_dev = None if v is None else torch.as_tensor(np.ascontiguousarray(v, dtype=np.float64), device="cuda").contiguous()

    @property
    def _K_inv(self):
        # materialised on first use: fit() no longer forms the inverse eagerly (gaussianprocess.py:317) because
        # batched predictions go through the factor (_mean_var)
        if self._Kinv_dev is None and self._L_dev is not None:
            self.set_K_inv()
        return None if self._Kinv_dev is None else self._Kinv_dev.cpu().numpy()

    @_K_inv.setter
    def _K_inv(self, v):
        self._Kinv_dev = None if v is None else torch.as_tensor(np.asarray(v, dtype=np.float64), device="cuda").contiguous()

    def __str__(self):
        s = f"------Gaussian Process Regression ({self.rank}/{self.size})------\n"
        s += "Kernel: {:s}".format(str(self.kernel))
        if hasattr(self, "train_x"):
            s += " {:d} energy ({:.5f})".format(self.N_energy, self.noise_e)
            s += " {:d} forces ({:.5f})\n".format(self.N_forces, self.noise_f)
        if self.use_base > 0:
            N1, N2, N3 = self.use_base, self.use_surrogate, self.fits
            s += "Total base/surrogate/gpr_fit calls: {}/{}/{}\n".format(N1, N2, N3)
        return s

    def todict(self):
        return {}

    def __repr__(self):
        return str(self)

    # ---------------------------------------------------------------------------------------------
    # device algebra
    # ---------------------------------------------------------------------------------------------
    def _n_energy_rows(self, train_x=None):
        train_x = self.train_x if train_x is None else train_x
        e = train_x.get('energy', [])
        if hasattr(e, "n_groups"):      # a device-resident Pack
            return e.n_groups
        if isinstance(e, tuple):
            return len(e[-1])
        return len(e)

    def _build_K(self, grad, f_tol=1e-10):
        """Training covariance (and dK/dl) on this device; row-block sharded when distributed.

        Returns (K [N, N], dK rows held by this rank or None, row ranges of those rows).
        Multi-GPU (replaces RBF_mb.py:471-521): every rank writes its energy / force row slabs of
        the full K in place (upper-triangle blocks only for K_ff), the slabs are all-gathered in
        place and the force-force block is mirrored; dK/dl stays local to the rank."""
        rank, size = gdist.world()
        e, f = packs_of(self.train_x)
        NE = e.n_groups if e is not None else 0
        NF = f.n_groups if f is not None else 0
        N = NE + 3 * NF
        if size == 1:
            K, dK = self.kernel.k_total_device(self.train_x, None, f_tol=f_tol, grad=grad)
            return K, dK, [(0, N)]
        from .device import build_energy_rows, build_force_rows
        args = self.kernel.cov_args(grad=grad, f_tol=f_tol)
        has_dk = args.pop("has_dk") and grad
        # force windows follow the measured throughput of the ranks (updated after every build)
        speed = getattr(self, "_shard_speed", None)
        if speed is None or len(speed) != size:
            speed = np.ones(size)
        f_rows = f.indices if f is not None else []
        windows = gdist.row_windows(e.indices if e is not None else [], f_rows, size, upper=True, speed=speed)
        (e0, e1), (f0, f1) = windows[rank]
        n_loc = (e1 - e0) + 3 * (f1 - f0)
        peer = self._peer_matrix(N)
        K = peer.tensor if peer is not None else torch.empty((N, N), dtype=F64, device="cuda")
        dK = None
        if has_dk:
            # one buffer with headroom for the whole optimisation: the adaptive windows change n_loc from build to build, and a
            # fresh multi-GB allocation per build (no cached block of exactly that size) costs tens of milliseconds
            buf = getattr(self, "_dK_buf", None)
            if buf is None or buf.shape[1] != N or buf.shape[0] < n_loc:
                self._dK_buf = buf = None
                buf = self._dK_buf = torch.empty((min(N, int(1.25 * n_loc) + 64), N), dtype=F64, device="cuda")
            dK = buf[:n_loc]
            dK.zero_()
        ff = dict(use_tol=args.pop("use_tol"), tol=args.pop("tol"), zeta_ff=args.pop("zeta_ff"))
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if peer is not None:
            # Fused gather (replaces the gather + bcast of RBF_mb.py:471-521): the K_fe / K_ff kernels store
            # every finished value into all ranks' copies of K over NVLink.  Every rank zeroes its own copy,
            # barrier (nobody still uses the previous K, all copies are zero), build, barrier (all stores landed).
            _zero_build_targets(K, NE)
            peer.barrier()
            Kee = torch.empty((NE, NE), dtype=F64, device="cuda")      # K_ee is small: NCCL gather of its row slabs
            build_energy_rows(side1=(e, f), side2=(e, f), window=(e0, e1), K=Kee[e0:e1],
                              dK=None if dK is None else dK[:e1 - e0], skip_kef=True, **args)
            t0.record()
            r0 = NE + 3 * f0
            slabs = [q for r, q in enumerate(gdist.slab_pointers(peer.ptrs, r0, 0, N)) if r != rank]
            build_force_rows(side1=(e, f), side2=(e, f), window=(f0, f1), K=K[r0:NE + 3 * f1],
                             dK=None if dK is None else dK[e1 - e0:], ff_mode=_lib.FF_UPPER, peer_slabs=slabs, **args, **ff)
            t1.record()
            if NE:
                gdist.gather_rows_inplace(Kee, [(w[0], (0, 0)) for w in windows], NE)
                K[:NE, :NE] = Kee
            peer.barrier()
        else:
            # energy rows: K_ee only; K_ef is the transpose of the K_fe rows the force windows produce
            build_energy_rows(side1=(e, f), side2=(e, f), window=(e0, e1), K=K[e0:e1],
                              dK=None if dK is None else dK[:e1 - e0], skip_kef=True, **args)
            t0.record()
            build_force_rows(side1=(e, f), side2=(e, f), window=(f0, f1), K=K[NE + 3 * f0:NE + 3 * f1],
                             dK=None if dK is None else dK[e1 - e0:], ff_mode=_lib.FF_UPPER, **args, **ff)
            t1.record()
            gdist.gather_rows_inplace(K, windows, NE)
        st = stream()
        if NF:
            _lib.call("gprb_symmetrize", c_vp(K.data_ptr() + (NE * N + NE) * 8), N, 3 * NF, st)
            if NE:
                _lib.call("gprb_transpose_copy", c_vp(K.data_ptr() + NE * 8), N, c_vp(K.data_ptr() + NE * N * 8), N,
                          3 * NF, NE, st)
            # re-balance: share of rank r ~ (cost it handled) / (time it took), damped
            t1.synchronize()
            rows = np.asarray(f_rows, dtype=np.float64)
            cost = rows * np.cumsum(rows[::-1])[::-1]
            mine = float(cost[f0:f1].sum()) / max(t0.elapsed_time(t1), 1e-3)
            rates = np.asarray(gdist.all_gather_floats(mine, device="cuda"))
            if np.all(rates > 0):
                self._shard_speed = 0.5 * speed / speed.sum() + 0.5 * rates / rates.sum()
            if os.environ.get("GPRB_DEBUG_SHARD"):
                print("[shard] rank %d window %d:%d kff %.1f ms speed %s" % (rank, f0, f1, t0.elapsed_time(t1),
                                                                          np.round(self._shard_speed, 4)), flush=True)
        return K, dK, [(e0, e1), (NE + 3 * f0, NE + 3 * f1)]

    def _peer_matrix(self, N):
        """This rank's peer-mapped copy of K for the fused gather (dist.PeerMatrix), or None: one is kept per
        GP and re-made (collectively) when the training set changes size."""
        rank, size = gdist.world()
        if size == 1 or size > _lib.MAX_DST or not gdist.peer_gather_enabled() or getattr(self, "_peer_failed", False):
            return None
        peer = getattr(self, "_peer", None)
        if peer is not None and peer.N != N:
            peer.close()
            peer = self._peer = None
        if peer is None:
            peer = self._peer = gdist.make_peer_matrix(N)
            if peer is None:
                self._peer_failed = True
        return peer

    def release_peer(self):
        """Collective: free the peer-mapped copy of K (every rank must call it)."""
        peer = getattr(self, "_peer", None)
        if peer is not None:
            peer.close()
            self._peer = None

    def _own(self, K):
        """A matrix the GP may keep: the peer-mapped K is overwritten by the next build, so copy out of it."""
        peer = getattr(self, "_peer", None)
        if peer is not None and peer.tensor is not None and K.data_ptr() == peer.tensor.data_ptr():
            return K.clone()
        return K

    def _factor(self, K, noise_e, noise_f):
        """K += noise; in-place Cholesky; alpha = K^-1 y.  Returns alpha (device vector)."""
        alpha, _ = self._lml_eval(K, None, [], noise_e, noise_f, want_grad=False)
        return alpha

    def set_K_inv(self):
        """K^-1 = L^-T L^-1 (gaussianprocess.py:128-131) on device: blocks of rows right of the diagonal by
        trailing-block triangular solves written in place (gprb_chol_inverse_rows, the route of the likelihood
        gradient: about 1.0 s instead of potri's 1.47 s at N = 32 980), then mirrored."""
        if self._Kinv_dev is None:
            N = self._L_dev.shape[0]
            Kinv = torch.empty((N, N), dtype=F64, device="cuda")
            st = stream()
            for (r0, r1, _) in _row_pieces([(0, N)], 0, N):
                _lib.call("gprb_chol_inverse_rows", ptr(self._L_dev), N, N, r0, r1, r0,
                          c_vp(Kinv.data_ptr() + (r0 * N + r0) * 8), N, st)
            _lib.call("gprb_symmetrize", ptr(Kinv), N, N, st)
            self._Kinv_dev = Kinv

    def log_marginal_likelihood(self, params, eval_gradient=False, clone_kernel=False):
        """
        Log marginal likelihood and (optionally) its gradient w.r.t. the hyper-parameters
        (GPML eq. 5.9; gaussianprocess.py:133-202).
        """
        require_cuda()
        if self.noise_bounds is None:
            noise_e, noise_f = self.noise_e, self.noise_f
            kernel_params = params
        else:
            noise_e = params[-1]
            noise_f = self.f_coef * noise_e
            kernel_params = params[:-1]
        kernel = self.kernel
        kernel.update(kernel_params)

        is_rbf = isinstance(kernel, RBF_mb)
        K, dK, r_ranges = self._build_K(grad=eval_gradient)
        N = K.shape[0]
        NE = self._n_energy_rows()
        if eval_gradient and is_rbf and gdist.world()[1] > 1:
            dK, r_ranges = self._rebalance_dK(dK, r_ranges, N, NE)
        try:
            _, out = self._lml_eval(K, dK if is_rbf else None, r_ranges, noise_e, noise_f,
                                    want_grad=eval_gradient, want_s0=not is_rbf)
        except _lib.NotPositiveDefinite:
            return (-np.inf, np.zeros_like(params)) if eval_gradient else -np.inf
        logdet, ya = out[0], out[1]
        MLL = -0.5 * ya - logdet - N / 2 * np.log(2 * np.pi)
        if not eval_gradient:
            return self._sync_ranks(MLL)
        if getattr(self, "_inverse_cost", None) is not None and gdist.world()[1] > 1:
            # re-balance the inverse-rows windows: share of rank r ~ (cost it handled) / (time its solves took), damped
            rates = np.asarray(gdist.all_gather_floats(self._inverse_cost / max(out[7], 1e-3), device="cuda"))
            if np.all(rates > 0):
                used = self._inverse_speed_used
                self._inverse_speed = 0.5 * used / used.sum() + 0.5 * rates / rates.sum()
            self._inverse_cost = None
        g_l, half_w_noise, half_w_base, g_s0 = out[2], out[3], out[4], out[5]
        if gdist.world()[1] > 1:
            g_l, half_w_noise, half_w_base, g_s0 = gdist.all_reduce_sum([g_l, half_w_noise, half_w_base, g_s0], device="cuda")
        if not is_rbf:
            # Dot: dK/dsigma0 = 0.8 * 2 sigma^2 sigma0 on the E-E block only (dot_kernel.py:58)
            g_s0 *= 0.8 * 2 * kernel.sigma ** 2 * kernel.sigma0
        # 1/2 tr(W (2/sigma) K0), K0 = K - noise:  tr(W K) = y.alpha - N
        g_sigma = ((ya - N) - 2.0 * half_w_noise) / kernel.sigma
        llg = np.array([g_sigma, g_l if is_rbf else g_s0, half_w_base])
        if self.noise_bounds is None:
            llg = llg[:-1]
        return self._sync_ranks(MLL, llg)

    def _rebalance_dK(self, dK, r_ranges, N, NE):
        """Re-cut the force rows of dK/dl over the ranks for the inverse-rows likelihood gradient.

        The covariance build balances n_I * sum_{J >= I} n_J (cost of the K_ff rows, ~ (N - r) per row); the trailing-block
        solves that follow cost (N - r)^2 per row, so the build's windows leave the first ranks with about twice the
        ideal solve time (SCALE_r01: 221 ms on rank 0 at 8 GPUs against 124 ms ideal).  dK/dl is only consumed by the
        traces, so its force rows are exchanged (one all-to-all over NVLink, about a third of the slab) into windows
        balanced for the solves; K is untouched."""
        rank, size = gdist.world()
        if dK is None or len(r_ranges) != 2:
            return dK, r_ranges
        (e0, e1), (r0, r1) = r_ranges
        NF = (N - NE) // 3
        first = NE + 3 * np.arange(NF, dtype=np.float64)
        cost = 3.0 * (N - first) ** 2
        # shares follow the measured solve throughput of the ranks (every block of rows also carries a fixed latency of two
        # triangular solves, which the flop model does not see): updated after every evaluation, identical on all ranks
        speed = getattr(self, "_inverse_speed", None)
        if speed is None or len(speed) != size:
            speed = np.ones(size)
        bounds = gdist.split_groups(cost, size, speed=speed)
        self._inverse_cost = float(cost[bounds[rank]:bounds[rank + 1]].sum())
        self._inverse_speed_used = speed
        f_old = gdist.all_gather_floats(float((r0 - NE) // 3), device="cuda") + [float(NF)]
        f_old = [int(v) for v in f_old]                      # force windows of the build, by rank (contiguous, ordered)
        # sanity: the build's windows tile [0, NF)
        if f_old[0] != 0 or any(f_old[k] > f_old[k + 1] for k in range(size)) or (r1 - NE) // 3 != f_old[rank + 1]:
            return dK, r_ranges
        ne_loc = e1 - e0
        send = [3 * max(0, min(f_old[rank + 1], bounds[d + 1]) - max(f_old[rank], bounds[d])) for d in range(size)]
        recv = [3 * max(0, min(f_old[s_ + 1], bounds[rank + 1]) - max(f_old[s_], bounds[rank])) for s_ in range(size)]
        g0, g1 = bounds[rank], bounds[rank + 1]
        n_new = ne_loc + 3 * (g1 - g0)
        buf = getattr(self, "_dK_inv_buf", None)          # reused across evaluations, like the build's buffer (_build_K)
        if buf is None or buf.shape[1] != N or buf.shape[0] < n_new:
            self._dK_inv_buf = buf = None
            buf = self._dK_inv_buf = torch.empty((min(N, int(1.25 * n_new) + 64), N), dtype=F64, device="cuda")
        new = buf[:n_new]
        if ne_loc:
            new[:ne_loc] = dK[:ne_loc]
        gdist.all_to_all_rows(new[ne_loc:], dK[ne_loc:], recv, send)
        return new, [(e0, e1), (NE + 3 * g0, NE + 3 * g1)]

    def _sync_ranks(self, lml, grad=None):
        """Every rank continues with rank 0's values (the reference broadcasts the parameters after each optimiser
        step, gaussianprocess.py:246-247, 305-306): the ranks' copies of K may differ in the last bit (summation order
        of row groups that straddle CTAs), and the host optimiser must take the same decisions on every rank or
        the ranks would issue different numbers of collective builds."""
        if gdist.world()[1] == 1:
            return lml if grad is None else (lml, grad)
        vals = gdist.broadcast_floats([lml] + ([] if grad is None else [float(g) for g in grad]), src=0, device="cuda")
        return vals[0] if grad is None else (vals[0], np.array(vals[1:]))

    def _lml_eval(self, K, dK, r_ranges, noise_e, noise_f, want_grad, want_s0=False):
        """gprb_lml_eval on the built covariance: noise, in-place Cholesky, alpha and the likelihood scalars with one
        host synchronisation (gaussianprocess.py:160-198 without the explicit inverse of :195).

        W = alpha alpha^T - K^-1 and dK/dl are symmetric, so tr(W dK) needs K^-1 only on and right of the
        diagonal, for the rows of dK this rank holds.  For a block of rows [r0, r1) that is K^-1[r0:r1, r0:N], a solve
        with the TRAILING block of the factor only (K^-1[T,T] = (L_TT L_TT^T)^-1), plus K^-1[0:NE, :] for the energy
        columns: the same 2 N^3 / 3 flops as potri but as large triangular solves, no N x N inverse buffer, and on G
        GPUs every rank solves only for its own rows.  Returns (alpha, the 8 scalars of gprb_lml_eval)."""
        N = K.shape[0]
        NE = self._n_energy_rows()
        y = torch.as_tensor(self.y_train[:, 0], device="cuda").contiguous()
        alpha = torch.empty(N, dtype=F64, device="cuda")
        out = (ctypes_double * 8)()
        flat = [int(v) for r in r_ranges for v in r]
        ranges = (ctypes.c_int * max(len(flat), 1))(*flat)
        parts = int(os.environ.get("GPRB_INVERSE_ROW_PARTS", "16"))
        # several GPUs: the factorisation is shared by the ranks (dist.distributed_cholesky) instead of repeated on each
        prefactored = 0
        if gdist.world()[1] > 1 and N >= self.DIST_CHOLESKY_MIN_N and os.environ.get("GPRB_DIST_CHOLESKY", "1") not in ("", "0"):
            _lib.call("gprb_add_noise", ptr(K), K.stride(0), N, NE, float(noise_e), float(noise_f), stream())
            info = gdist.distributed_cholesky(K, nb=int(os.environ.get("GPRB_DIST_CHOLESKY_NB", "1024")))
            if info != 0:
                raise _lib.NotPositiveDefinite(_lib.ERR_LINALG, "matrix not positive definite (distributed potrf info = %d)" % info)
            prefactored = 1
        n_work = int(_lib.load().gprb_lml_eval_work(N, NE, int(bool(want_grad)), parts))
        work = torch.empty(max(n_work, 1), dtype=F64, device="cuda")        # torch's caching allocator keeps it across evaluations
        _lib.call("gprb_lml_eval", ptr(K), K.stride(0), N, NE, ptr(y), float(noise_e), float(noise_f),
                  ptr(dK), dK.stride(0) if dK is not None else N, len(r_ranges), ranges, int(bool(want_grad)),
                  int(bool(want_s0)), parts, prefactored, ptr(alpha), ptr(work), n_work, out, stream())
        return alpha, [float(v) for v in out]

    def optimize(self, fun, theta0, bounds, maxiter=10):
        """L-BFGS-B on the host, identical options to gaussianprocess.py:215-219."""
        opt_res = minimize(fun, theta0, method="L-BFGS-B", bounds=bounds, jac=True,
                           options={'maxiter': maxiter, 'ftol': 1e-2})
        return opt_res.x, opt_res.fun

    def fit(self, TrainData=None, show=True, opt=True, maxiter=10):
        """
        Fit the GPR model (gaussianprocess.py:222-317).

        Args:
            TrainData: a dictionary of energy/force/db data
            show: print the information or not
            opt: optimize the hyperparameters or not
            maxiter: maximum number of L-BFGS-B iterations
        """
        require_cuda()
        if TrainData is None:
            self.update_y_train()
        else:
            self.set_train_pts(TrainData)

        if self.rank == 0 and show:
            print(self)

        def obj_func(params, eval_gradient=True):
            if eval_gradient:
                lml, grad = self.log_marginal_likelihood(params, eval_gradient=True, clone_kernel=False)
                if show:
                    strs = "Loss: {:12.3f} ".format(-lml)
                    for para in params:
                        strs += "{:6.3f} ".format(para)
                    if self.rank == 0:
                        print(strs)
                        self.logging.info(strs)
                return (-lml, -grad)
            lml = self.log_marginal_likelihood(params, clone_kernel=False)
            return -lml

        hyper_params = self.kernel.parameters()
        hyper_bounds = list(self.kernel.bounds)
        if self.noise_bounds is not None:
            hyper_params += [self.noise_e]
            hyper_bounds += [self.noise_bounds]

        if opt:
            if self.rank == 0:
                print(f"Update GP model => {self.N_queue}/{maxiter}")
            params, _ = self.optimize(obj_func, hyper_params, hyper_bounds, maxiter=maxiter)
            if gdist.world()[1] > 1:       # params = comm.bcast(params, root=0), gaussianprocess.py:305-306
                params = np.array(gdist.broadcast_floats(params, src=0, device="cuda"))
            if self.noise_bounds is not None:
                self.kernel.update(params[:-1])
                self.noise_e = params[-1]
                self.noise_f = self.f_coef * params[-1]
            else:
                self.kernel.update(params)

        # final covariance with the pair-cut variant of K_ff (f_tol = 1e-10), as k_total at :286
        K, _, _ = self._build_K(grad=False)
        K = self._own(K)
        self._alpha_dev = self._factor(K, self.noise_e, self.noise_f)
        self._L_dev = K
        self.logging.info("Cholesky Decomp is Complete")
        self._Kinv_dev = None

        self.N_energy_queue = 0
        self.N_forces_queue = 0
        self.N_queue = 0
        self.fits += 1
        # set_K_inv() of gaussianprocess.py:317 is deferred to the first consumer of the explicit inverse
        # (single-structure variance, return_cov, the _K_inv attribute): see _mean_var

    def _predict_device(self, X, train_x, f_tol, return_std):
        """K* on device, mean and variance (gaussianprocess.py:338, 368-377 / 880, 904-908)."""
        e, f = packs_of(X)                       # packed once, shared by K* and the prior variance
        Xp = {}
        if e is not None:
            Xp["energy"] = e
        if f is not None:
            Xp["force"] = f
        K_trans, _ = self.kernel.k_total_device(Xp, train_x, f_tol=f_tol, grad=False)
        diag = None
        if return_std:
            diag = self.kernel.diag_device(X if isinstance(self.kernel, Dot_mb) else Xp, _packed_ok=True)
        mean, var = self._mean_var(K_trans, diag)
        return K_trans, mean, var

    # Variance routes.  The reference multiplies K* with the explicit inverse (gaussianprocess.py:369, 905: "inverse",
    # gprb_predict: half product of the symmetric inverse, m N^2 flops); |L^-1 k*|^2 through the Cholesky factor ("chol",
    # gprb_predict_chol: one trsm, m N^2 flops, no N x N inverse to form) is algebraically the same number.
    # Which one tracks the reference?  Measured on real Cu32 rows at N = 2 328, cond(K) = 4e8, sigma = 4e-4 .. 3e-2
    # (tests/test_gpu_gp.py::test_sigma_routes_against_reference_formula, profiles/r02_sigma_routes.txt), max |d sigma|:
    #     the reference's own formula (numpy / LAPACK, explicit inverse) vs an iteratively refined value   4.0e-7
    #     device "chol" route  vs the refined value   1.6e-13        vs the reference's formula   4.0e-7
    #     device "inverse" route vs the refined value 1.3e-6         vs the reference's formula   8.8e-7
    # i.e. the explicit-inverse arithmetic loses cond(K) eps in the cancellation diag - k*^T K^-1 k* wherever it runs, two
    # implementations of it differ from each other by MORE than either differs from the factor route, and the factor route
    # is exact to rounding.  So batches take the factor route (closest to the truth AND to the reference's numbers); below
    # CHOL_VARIANCE_MIN_ROWS rows of K* (single structures: a triangular solve with few right-hand sides is latency bound,
    # 15 ms vs 4 ms at N = 32 980) the reference's explicit-inverse formula is used.  GPRB_VARIANCE_ROUTE = chol | inverse
    # forces one route; variance_route_probe() reports how far the two are apart on the current model.
    CHOL_VARIANCE_MIN_ROWS = 512
    PROBE_ROWS = 128
    DIST_CHOLESKY_MIN_N = 8192          # below this the panels are too small to pay for their broadcasts

    def variance_route_probe(self, K_trans, diag):
        """max |sigma_chol - sigma_inverse| over the first PROBE_ROWS rows of K*: a direct estimate of the conditioning
        error of the explicit-inverse variance formula (the reference's) on the fitted model.  Diagnostic only."""
        m, N = min(K_trans.shape[0], self.PROBE_ROWS), K_trans.shape[1]
        Kp, dp = K_trans[:m], diag[:m]
        mean, work = torch.empty(m, dtype=F64, device="cuda"), torch.empty((m, N), dtype=F64, device="cuda")
        v_c, v_i = torch.empty(m, dtype=F64, device="cuda"), torch.empty(m, dtype=F64, device="cuda")
        self.set_K_inv()
        _lib.call("gprb_predict_chol", m, N, ptr(Kp), K_trans.stride(0), ptr(self._alpha_dev), ptr(self._L_dev), N,
                  ptr(dp), ptr(mean), ptr(v_c), ptr(work), stream())
        _lib.call("gprb_predict", m, N, ptr(Kp), K_trans.stride(0), ptr(self._alpha_dev), ptr(self._Kinv_dev), N,
                  ptr(dp), ptr(mean), ptr(v_i), ptr(work), stream())
        return float((torch.sqrt(v_c) - torch.sqrt(v_i)).abs().max())

    def _mean_var(self, K_trans, diag):
        """mean = K* alpha and, when `diag` (the prior variances) is given, var = max(diag - k*^T K^-1 k*, 0)."""
        m, N = K_trans.shape
        mean = torch.empty(m, dtype=F64, device="cuda")
        if diag is None:
            _lib.call("gprb_predict", m, N, ptr(K_trans), K_trans.stride(0), ptr(self._alpha_dev), c_vp(0), N, c_vp(0), ptr(mean),
                      c_vp(0), c_vp(0), stream())
            return mean, None
        var = torch.empty(m, dtype=F64, device="cuda")
        work = torch.empty((m, N), dtype=F64, device="cuda")
        route = os.environ.get("GPRB_VARIANCE_ROUTE", "auto")          # auto | chol | inverse
        if self._L_dev is not None and (route == "chol" or (route == "auto" and m >= self.CHOL_VARIANCE_MIN_ROWS)):
            _lib.call("gprb_predict_chol", m, N, ptr(K_trans), K_trans.stride(0), ptr(self._alpha_dev), ptr(self._L_dev), N,
                      ptr(diag), ptr(mean), ptr(var), ptr(work), stream())
        else:
            self.set_K_inv()
            _lib.call("gprb_predict", m, N, ptr(K_trans), K_trans.stride(0), ptr(self._alpha_dev), ptr(self._Kinv_dev), N,
                      ptr(diag), ptr(mean), ptr(var), ptr(work), stream())
        return mean, var

    def predict(self, X, stress=False, total_E=False, return_std=False, return_cov=False):
        """
        Predict energy/force rows for packed or listed data `X` (gaussianprocess.py:319-379).
        """
        require_cuda()
        train_x = self.get_train_x()
        if stress:
            # gaussianprocess.py:331-333: K* from k_total_with_stress, the stress rows themselves are discarded
            K_trans, _ = self.kernel.k_total_stress_device(X, train_x)
            return_std = return_cov = False
            mean, var = self._mean_var(K_trans, None)
        else:
            K_trans, mean, var = self._predict_device(X, train_x, 1e-10, return_std and not return_cov)
        y_mean = mean.cpu().numpy()

        Npts = 0
        if 'energy' in X:
            Npts += len(X["energy"][-1]) if isinstance(X["energy"], tuple) else len(X["energy"])
        if 'force' in X:
            Npts += 3 * len(X["force"][-1]) if isinstance(X["force"], tuple) else 3 * len(X["force"])
        factors = np.ones(Npts)
        if total_E:
            if isinstance(X["energy"], tuple):
                N_atoms = np.array([x for x in X["energy"][-1]])
            else:
                N_atoms = np.array([len(x) for x in X["energy"]])
            factors[:len(N_atoms)] = N_atoms
        y_mean *= factors

        if return_cov:
            # y_cov = k(X, X) - K* K^-1 K*^T with v = cho_solve(L, K*^T)   (:363-366)
            y_cov, _ = self.kernel.k_total_device(X, None, grad=False)
            m_, N_ = K_trans.shape
            work = torch.empty((m_, N_), dtype=F64, device="cuda")
            _lib.call("gprb_predict_cov", m_, N_, ptr(K_trans), K_trans.stride(0), ptr(self._L_dev), N_, ptr(y_cov), y_cov.stride(0),
                      ptr(work), stream())
            return y_mean, y_cov.cpu().numpy()
        elif return_std:
            return y_mean, np.sqrt(var.cpu().numpy()) * factors
        return y_mean

    # ---------------------------------------------------------------------------------------------
    # training-set bookkeeping (host; identical semantics to gaussianprocess.py:381-629)
    # ---------------------------------------------------------------------------------------------
    def set_train_pts(self, data, mode="w"):
        """Set ("w") or append ("a+") training points from {'energy','force','db'} lists (:381-425)."""
        if mode == "w" or self.train_x is None:
            self.train_x = {'energy': [], 'force': []}
            self.train_y = {'energy': [], 'force': []}
            self.train_db = []

        N_E, N_F = 0, 0
        for d in data["db"]:
            (atoms, energy, force, energy_in, force_in) = d
            if energy_in:
                e_id = N_E + 1
                N_E += 1
            else:
                e_id = None
            if len(force_in) > 0:
                f_ids = [N_F + i for i in range(len(force_in))]
                N_F += len(force_in)
            else:
                f_ids = []
            self.train_db.append((atoms, energy, force, energy_in, force_in, e_id, f_ids))

        for key in data.keys():
            if key == 'energy' and len(data[key]) > 0:
                self.add_train_pts_energy(data[key])
            elif key == 'force' and len(data[key]) > 0:
                self.add_train_pts_force(data[key])

        self.update_y_train()
        self.N_energy += N_E
        self.N_forces += N_F
        self.N_energy_queue += N_E
        self.N_forces_queue += N_F
        self.N_queue += N_E + N_F

    def remove_train_pts(self, e_ids, f_ids):
        """Delete training points and refit (:427-464)."""
        data = {"energy": [], "force": [], "db": []}
        energy_data = tuple_to_list(self.train_x['energy'], mode='energy')
        force_data = tuple_to_list(self.train_x['force'])
        for i, (X, ele) in enumerate(energy_data):
            if i not in e_ids:
                data['energy'].append((X, self.train_y['energy'][i], ele))
        for i, (X, dxdr, ele) in enumerate(force_data):
            if i not in f_ids:
                data["force"].append((X, dxdr, self.train_y['force'][i], ele))
        for (atoms, energy, force, energy_in, force_in, e_id, _f_ids) in self.train_db:
            if e_id in e_ids:
                energy_in = False
            _force_in = [force_in[i] for i, f_id in enumerate(_f_ids) if f_id not in f_ids]
            if energy_in or len(_force_in) > 0:
                data['db'].append((atoms, energy, force, energy_in, _force_in))
        self.N_energy = self.N_forces = 0
        self.N_energy_queue = self.N_forces_queue = self.N_queue = 0
        self.set_train_pts(data)
        self.fit()

    def compute_base_potential(self, atoms):
        return self.base_potential.calculate(atoms)

    def update_y_train(self):
        """Targets as one column: per-atom energies, then (Fx, Fy, Fz) per force centre (:472-488)."""
        E = np.asarray(self.train_y["energy"], dtype=np.float64).reshape(-1)
        F = np.asarray(self.train_y["force"], dtype=np.float64).reshape(-1)
        self.y_train = np.concatenate((E, F)).reshape(-1, 1)

    def validate_data(self, test_data=None, total_E=False, return_std=False, show=False):
        """Predict a labelled data set (default: the training set) (:490-535)."""
        if test_data is None:
            test_X_E = {"energy": self.train_x['energy']}
            test_X_F = {"force": self.train_x['force']}
            NE = len(test_X_E['energy'][-1]) if len(test_X_E['energy']) > 0 else 0
            E = self.y_train[:NE].flatten()
            F = self.y_train[NE:].flatten()
        else:
            test_X_E = {"energy": [(data[0], data[2]) for data in test_data['energy']]}
            test_X_F = {"force": [(data[0], data[1], data[3]) for data in test_data['force']]}
            E = np.array([data[1] for data in test_data['energy']])
            F = np.array([data[2] for data in test_data['force']]).flatten()

        if total_E:
            for i in range(len(E)):
                E[i] *= len(test_X_E['energy'][i])

        E_Pred, E_std, F_Pred, F_std = None, None, None, None
        if return_std:
            if len(test_X_E['energy']) > 0:
                E_Pred, E_std = self.predict(test_X_E, total_E=total_E, return_std=True)
            if len(test_X_F['force']) > 0:
                F_Pred, F_std = self.predict(test_X_F, return_std=True)
            if show:
                self.update_error(E, E_Pred, F, F_Pred)
            return E, E_Pred, E_std, F, F_Pred, F_std
        if len(test_X_E['energy']) > 0:
            E_Pred = self.predict(test_X_E, total_E=total_E)
        if len(test_X_F['force']) > 0:
            F_Pred = self.predict(test_X_F)
        if show:
            self.update_error(E, E_Pred, F, F_Pred)
        return E, E_Pred, F, F_Pred

    def update_error(self, E, E_Pred, F, F_Pred):
        e_r2, e_mae, e_rmse = metric_values(E, E_Pred)
        f_r2, f_mae, f_rmse = metric_values(F, F_Pred)
        self.error = {"energy_r2": e_r2, "energy_mae": e_mae, "energy_rmse": e_rmse,
                      "forces_r2": f_r2, "forces_mae": f_mae, "forces_rmse": f_rmse}
        if self.rank == 0:
            for key in self.error.keys():
                self.logging.info(f"{key:<12s}: {self.error[key]:.4f}")

    def get_train_x(self):
        """Training data without the not-yet-fitted queue (:553-577)."""
        if self.N_queue > 0:
            train_x = {}
            (_X, _ELE, _indices) = self.train_x['energy']
            NE = self.N_energy - self.N_energy_queue
            if NE > 0:
                ids = sum(_indices[:NE])
                train_x['energy'] = (_X[:ids], _ELE[:ids], _indices[:NE])
            else:
                train_x['energy'] = (_X, _ELE, _indices)
            NF = self.N_forces - self.N_forces_queue
            (_X, _dXdR, _ELE, _indices) = self.train_x['force']
            if NF > 0:
                ids = sum(_indices[:NF])
                train_x['force'] = (_X[:ids], _dXdR[:ids], _ELE[:ids], _indices[:NF])
            else:
                train_x['force'] = (_X, _dXdR, _ELE, _indices)
            return train_x
        return self.train_x

    def add_train_pts_energy(self, energy_data):
        """Append (x, E/atom, ele) items to the packed energy set (:579-600)."""
        (X, ELE, indices, E) = list_to_tuple(energy_data, include_value=True, mode='energy')
        if len(self.train_x['energy']) == 3:
            (_X, _ELE, _indices) = self.train_x['energy']
            self.train_x['energy'] = (np.concatenate((_X, X), axis=0), np.concatenate((_ELE, ELE), axis=0),
                                      list(_indices) + list(indices))
            self.train_y['energy'] = list(self.train_y['energy']) + list(E)
        else:
            self.train_x['energy'] = (X, ELE, indices)
            self.train_y['energy'] = E

    def add_train_pts_force(self, force_data):
        """Append (x, dxdr, F, ele) items to the packed force set (:602-629)."""
        (X, dXdR, ELE, indices, F) = list_to_tuple(force_data, include_value=True)
        if len(self.train_x['force']) == 4:
            (_X, _dXdR, _ELE, _indices) = self.train_x['force']
            self.train_x['force'] = (np.concatenate((_X, X), axis=0), np.concatenate((_dXdR, dXdR), axis=0),
                                     np.concatenate((_ELE, ELE), axis=0), list(_indices) + list(indices))
            self.train_y['force'] = list(self.train_y['force']) + list(F)
        else:
            self.train_x['force'] = (X, dXdR, ELE, indices)
            self.train_y['force'] = F

    # ---------------------------------------------------------------------------------------------
    # persistence: json model file + ASE sqlite database (SURVEY.md §8f #2)
    # ---------------------------------------------------------------------------------------------
    def save_dict(self, db_filename):
        noise = {"energy": self.noise_e, "force": self.noise_f, "f_coef": self.f_coef, "bounds": self.noise_bounds}
        dict0 = {"noise": noise, "kernel": self.kernel.save_dict(), "descriptor": self.descriptor.save_dict(),
                 "db_filename": db_filename}
        if self.error is not None:
            dict0["error"] = self.error
        if self.base_potential is not None:
            dict0["base_potential"] = self.base_potential.save_dict()
        return dict0

    def save(self, filename, db_filename, verbose=True):
        with open(filename, "w") as fp:
            json.dump(self.save_dict(db_filename), fp, indent=4)
        self.export_ase_db(db_filename, permission="w")
        if verbose:
            print(f"save model to {filename} and {db_filename}")

    def export_ase_db(self, db_filename, permission="w"):
        """Write the training structures and their labels to an ASE sqlite database
        (gaussianprocess.py:689-724).  The rows are written by gpr_calculator_b200.asedb (ASE's own
        file layout), so ASE is not needed and the file can be opened with ase.db.connect."""
        from . import asedb
        rows = []
        for (struc, energy, force, energy_in, force_in, _, _) in self.train_db:
            actual_energy, actual_forces = deepcopy(energy), np.array(force, dtype=float)
            if self.base_potential is not None:
                energy_off, force_off, _ = self.compute_base_potential(struc)
                actual_energy += energy_off
                actual_forces += force_off
            data = {"energy": float(energy), "force": np.asarray(force, dtype=np.float64), "energy_in": bool(energy_in),
                    "force_in": [int(i) for i in force_in]}
            kvp = {"dft_energy": float(actual_energy) / len(force), "dft_fmax": float(np.max(np.abs(actual_forces.flatten())))}
            rows.append((struc, kvp, data))
        asedb.write_rows(db_filename, rows, append=(permission != "w"))

    @classmethod
    def load(cls, filename, N_max=None, device='cuda'):
        with open(filename, "r") as fp:
            dict0 = json.load(fp)
        instance = cls.load_from_dict(dict0, device=device)
        instance.extract_db(dict0["db_filename"], N_max)
        if instance.rank == 0:
            print(f"load GP model from {filename}")
            print(instance)
        return instance

    def extract_db(self, db_filename, N_max=None, batch=16):
        """Rebuild the training set from an ASE database (gaussianprocess.py:726-821): the descriptors
        of all structures are recomputed, `batch` structures per device pass (the reference recomputes
        them one by one, split over MPI ranks)."""
        from . import asedb
        rows = []
        for n, row in enumerate(asedb.read_rows(db_filename)):
            if N_max is not None and n >= N_max:
                break
            rows.append(row)
        pts = {"energy": [], "force": [], "db": []}
        for s0 in range(0, len(rows), batch):
            part = rows[s0:s0 + batch]
            atoms_list = [r.toatoms() for r in part]
            if hasattr(self.descriptor, "calculate_batch"):
                descs = self.descriptor.calculate_batch(atoms_list, to_host=True)
            else:
                descs = [self.descriptor.calculate(a) for a in atoms_list]
            for row, atoms, d in zip(part, atoms_list, descs):
                energy, force = float(row.data["energy"]), np.array(row.data["force"], dtype=float)
                energy_in, force_in = bool(row.data["energy_in"]), [int(i) for i in row.data["force_in"]]
                ele = atomic_numbers(d['elements'])
                if energy_in:
                    pts["energy"].append((d['x'], energy / len(atoms), ele))
                for i in force_in:
                    x, dxdr, e = force_rows(d, ele, i)
                    pts["force"].append((x, dxdr, force[i], e))
                pts["db"].append((atoms, energy, force, energy_in, force_in))
        self.N_energy = self.N_forces = 0
        self.N_energy_queue = self.N_forces_queue = self.N_queue = 0
        self.set_train_pts(pts, "w")

    # ---------------------------------------------------------------------------------------------
    # structure-level API
    # ---------------------------------------------------------------------------------------------
    def _get_fixed_atoms(self, struc):
        """Indices held by a FixAtoms-like constraint (anything exposing get_indices) (:823-832)."""
        for c in getattr(struc, "constraints", []) or []:
            if type(c).__name__ == "FixAtoms" and hasattr(c, "get_indices"):
                return list(c.get_indices())
        return []

    def predict_structure(self, struc, stress=True, return_std=False, f_tol=1e-8):
        """
        Energy, forces (and their standard deviations) of one structure (:834-918).

        stress=True (the reference's default) needs a descriptor created with stress=True; every atom is
        then a force centre (gaussianprocess.py:862-864) and S is the per-atom stress [n_atoms, 6] in the
        order xx, yy, zz, xy, xz, yz (:890-891).  GPR.calculate passes stress=False by default
        (calculator.py:124-127).
        """
        require_cuda()
        if stress:
            return self._predict_structure_stress(struc, return_std, f_tol)
        fix_ids = set(self._get_fixed_atoms(struc))
        free_ids = [i for i in range(len(struc)) if i not in fix_ids]
        if hasattr(self.descriptor, "calculate_batch"):
            # descriptors stay on the device: rows are gathered there (batch.rows_from_batch)
            from .batch import rows_from_batch
            E_t, F_t = rows_from_batch(self.descriptor.calculate_batch([struc], to_host=False), [free_ids])
            data = {"energy": E_t}
            if F_t is not None:
                data["force"] = F_t
        else:
            d = self.descriptor.calculate(struc, use_mpi=True)
            ele = atomic_numbers(d['elements'])
            data = {"energy": list_to_tuple([(d['x'], ele)], mode='energy')}
            if len(free_ids) > 0:
                data["force"] = [force_rows(d, ele, i) for i in free_ids]

        train_x = self.get_train_x()
        _, mean, var = self._predict_device(data, train_x, f_tol, return_std)
        y_mean = mean.cpu().numpy()
        y_mean[0] *= len(struc)
        E = y_mean[0]
        F = np.zeros((len(struc), 3))
        F[free_ids] = y_mean[1:].reshape([len(free_ids), 3])
        S = None

        if self.base_potential is not None:
            energy_off, force_off, _ = self.compute_base_potential(struc)
            E += energy_off
            F += force_off

        if return_std:
            y_std = np.sqrt(var.cpu().numpy())
            E_std = y_std[0]
            F_std = np.zeros((len(struc), 3))
            F_std[free_ids] = y_std[1:].reshape([len(free_ids), 3])
            return E, F, S, E_std, F_std
        return E, F, S

    def _predict_structure_stress(self, struc, return_std, f_tol):
        """predict_structure(stress=True): K* rows of the energy, of all 3 n force components and of the
        6 n Voigt stress components (k_total_with_stress), mean = K* alpha."""
        from .batch import rows_from_batch
        from .device import energy_pack, stress_packs
        if not getattr(self.descriptor, "stress", False) or not hasattr(self.descriptor, "calculate_batch"):
            raise ValueError("predict_structure(stress=True) needs a descriptor created with stress=True "
                             "(the reference reads d['rdxdr'], gaussianprocess.py:862)")
        n = len(struc)
        fixed = set(self._get_fixed_atoms(struc))
        free_ids = [i for i in range(n) if i not in fixed]
        E_t, F_t = rows_from_batch(self.descriptor.calculate_batch([struc], to_host=False), None, stress=True)
        e1, (f1, sa, sb) = energy_pack(E_t), stress_packs(F_t)
        train_x = self.get_train_x()
        K, K1 = self.kernel.k_total_stress_device({"energy": e1, "force": (f1, sa, sb)}, train_x, tol=f_tol)
        diag = None
        if return_std:
            diag = self.kernel.diag_device({"energy": E_t, "force": (F_t[0], F_t[1][:, :, :3].contiguous(), F_t[2], F_t[3])}
                                           if isinstance(self.kernel, Dot_mb) else {"energy": e1, "force": f1}, _packed_ok=True)
        mean, var = self._mean_var(K, diag)
        y_mean = mean.cpu().numpy()
        E = y_mean[0] * n
        F_all = y_mean[1:].reshape(n, 3)
        F = np.zeros((n, 3))
        F[free_ids] = F_all[free_ids]
        S = self._mean_var(K1, None)[0].cpu().numpy().reshape(n, 6)
        if self.base_potential is not None:
            energy_off, force_off, stress_off = self.compute_base_potential(struc)
            E += energy_off
            F += force_off
            S += stress_off
        if return_std:
            y_std = np.sqrt(var.cpu().numpy())
            F_std = np.zeros((n, 3))
            F_std[free_ids] = y_std[1:].reshape(n, 3)[free_ids]
            return E, F, S, y_std[0], F_std
        return E, F, S

    def predict_structures(self, strucs, return_std=False, f_tol=1e-8, batch=32, shard=True):
        """Batched predict_structure(stress=False): descriptors, K*, mean and variance of `batch`
        structures per device pass (the "predict 10k structures" path of the benchmark).

        Multi-GPU (torch.distributed initialised, every rank holds the fitted model and calls this with the same
        list): the structures are sharded over the ranks in contiguous blocks balanced by atom count, every rank
        predicts its block and the results are combined with one all-reduce of a [sum(1 + 3 n) x (1 or 2)] buffer in
        which each rank fills only its own slots (replaces the reference's per-structure rank-0 evaluation + bcast,
        gaussianprocess.py:834-918 under mpi4py).  shard=False: every rank predicts the whole list (replicas).

        Returns a list of (E, F, None) or (E, F, None, E_std, F_std) tuples, one per structure, equal to
        what predict_structure returns for each of them."""
        require_cuda()
        if self.base_potential is not None:
            raise NotImplementedError("base potentials are outside the B200 hot path")
        rank, size = gdist.world()
        if size == 1 or not shard or len(strucs) == 0:
            return self._predict_structures_local(strucs, return_std, f_tol, batch)
        bounds = gdist.split_groups([len(s_) for s_ in strucs], size)
        mine = self._predict_structures_local(strucs[bounds[rank]:bounds[rank + 1]], return_std, f_tol, batch)
        return gdist.gather_predictions(mine, [len(s_) for s_ in strucs], bounds[rank], return_std, device="cuda")

    def _predict_structures_local(self, strucs, return_std, f_tol, batch):
        from .batch import rows_from_batch
        train_x = self.get_train_x()
        out = []
        for s0 in range(0, len(strucs), batch):
            part = strucs[s0:s0 + batch]
            free = []
            for st_ in part:
                fixed = set(self._get_fixed_atoms(st_))
                free.append([i for i in range(len(st_)) if i not in fixed])
            E_t, F_t = rows_from_batch(self.descriptor.calculate_batch(part, to_host=False), free)
            data = {"energy": E_t}
            if F_t is not None:
                data["force"] = F_t
            _, mean, var = self._predict_device(data, train_x, f_tol, return_std)
            y = mean.cpu().numpy()
            sd = np.sqrt(var.cpu().numpy()) if return_std else None
            pos = len(part)
            for k, st_ in enumerate(part):
                n, nf = len(st_), len(free[k])
                F = np.zeros((n, 3))
                F[free[k]] = y[pos:pos + 3 * nf].reshape(nf, 3)
                if return_std:
                    F_std = np.zeros((n, 3))
                    F_std[free[k]] = sd[pos:pos + 3 * nf].reshape(nf, 3)
                    out.append((y[k] * n, F, None, sd[k], F_std))
                else:
                    out.append((y[k] * n, F, None))
                pos += 3 * nf
        return out

    def add_structure(self, data, N_max=20, tol_e_var=1.2, tol_f_var=1.2, add_force=True):
        """
        Add training points from a labelled structure (:921-1002): the energy always; up to N_max
        force centres whose predicted std or error exceeds the tolerance and whose descriptor is
        new (utilities.new_pt).
        """
        tol_e_var *= self.noise_e
        tol_f_var *= self.noise_f
        pts_to_add = {"energy": [], "force": [], "db": []}
        (atoms, energy, force) = data

        if self.base_potential is not None:
            energy_off, force_off, _ = self.compute_base_potential(atoms)
        else:
            energy_off, force_off = 0, np.zeros((len(atoms), 3))
        energy = energy - energy_off
        force = force - force_off
        my_data = convert_train_data([(atoms, energy, force)], self.descriptor)

        if self._alpha_dev is not None:
            E, E1, E_std, F, F1, F_std = self.validate_data(my_data, return_std=True)
            E_std = E_std[0]
            F_std = F_std.reshape((len(atoms), 3))
        else:
            E = E1 = [energy / len(atoms)]
            F = F1 = force.flatten()
            E_std = 2 * tol_e_var
            F_std = 2 * tol_f_var * np.ones((len(atoms), 3))
        # NOTE: F and F1 stay FLAT (3n,) and are indexed by atom id below, exactly as the reference
        # does (gaussianprocess.py:979) — this decides which force centres enter the training set.
        F, F1 = np.asarray(F), np.asarray(F1)

        pts_to_add["energy"] = my_data["energy"]
        N_energy, energy_in = 1, True

        force_in = []
        if add_force:
            xs_added = []
            for f_id in range(len(atoms)):
                include = False
                if np.max(F_std[f_id]) > tol_f_var or np.max(abs(F[f_id] - F1[f_id])) > 1.5 * tol_f_var:
                    X = my_data["energy"][0][0][f_id]
                    _ele = my_data["energy"][0][2][f_id]
                    if len(xs_added) == 0 or new_pt((X, _ele), xs_added):
                        include = True
                if include:
                    force_in.append(f_id)
                    xs_added.append((X, _ele))
                    pts_to_add["force"].append(my_data["force"][f_id])
                if len(force_in) == N_max:
                    break

        N_pts = N_energy + len(force_in)
        if N_pts > 0:
            pts_to_add["db"].append((atoms, energy, force, energy_in, force_in))
            self.set_train_pts(pts_to_add, mode="a+")
        errors = (E[0] + energy_off, E1[0] + energy_off, E_std,
                  F + force_off.flatten(), F1 + force_off.flatten(), F_std)
        return pts_to_add, N_pts, errors

    def sparsify(self, e_tol=1e-10, f_tol=1e-10):
        """Drop training points in the near-null space of K (CUR, gaussianprocess.py:1004-1023).  K stays on
        the device: eigen-decomposition by cuSOLVER syevd and leverage scores in gprb_cur_scores; the
        O(N_f^2) Python double loop of the reference is a vectorised membership test."""
        require_cuda()
        K, _ = self.kernel.k_total_device(self.train_x, None, grad=False)
        N_e = len(self.train_x["energy"][-1])
        N_f = len(self.train_x["force"][-1])
        pts_e = CUR_device(K[:N_e, :N_e], e_tol)
        pts = CUR_device(K[N_e:, N_e:], f_tol)
        pts_f = []
        if N_f > 1:
            hit = np.zeros(3 * N_f, dtype=bool)
            hit[pts] = True
            pts_f = [int(i) for i in np.flatnonzero(hit.reshape(N_f, 3).all(axis=1))]
        pts_e = [int(i) for i in pts_e]
        print("{:d} energy and {:d} forces will be removed".format(len(pts_e), len(pts_f)))
        if len(pts_e) + len(pts_f) > 0:
            self.remove_train_pts(pts_e, pts_f)

    @classmethod
    def set_GPR(cls, images, base, kernel='RBF',
                zeta=2.0, noise_e=0.002, noise_f=0.1,
                lmax=4, nmax=3, rcut=5.0, json_file=None,
                overwrite=False):
        """Set up and train a GPR model from images with a base calculator (:1025-1072)."""
        if json_file is not None and os.path.exists(json_file):
            instance = cls.load(json_file)
            if overwrite:
                instance.noise_e = noise_e
                instance.noise_f = noise_f
                if instance.kernel.name != kernel:
                    if kernel == "RBF":
                        instance.kernel = RBF_mb(para=[1.0, 0.1], zeta=zeta)
                    else:
                        instance.kernel = Dot_mb(para=[2, 2.0], zeta=zeta)
            instance.fit()
            instance.set_K_inv()
        else:
            instance = cls(kernel=None, descriptor=None, base_potential=None)
            if kernel == 'Dot':
                instance.kernel = Dot_mb(para=[2, 2.0], zeta=zeta)
            else:
                instance.kernel = RBF_mb(para=[1.0, 0.1], zeta=zeta)
            instance.descriptor = _lazy_SO3()(nmax=nmax, lmax=lmax, rcut=rcut)
            instance.noise_e = noise_e
            instance.noise_f = noise_f
            instance.train_images(images, base)
        return instance

    def train_images(self, images, base):
        """Label the images with the base calculator, add them and fit (:1074-1116)."""
        for i, image in enumerate(images):
            image.calc = base
            if hasattr(image.calc, 'set'):
                image.calc.set(directory=f"GP/calc_{i}")
            eng = image.get_potential_energy()
            forces = image.get_forces()
            if self.rank == 0:
                print(f"Calculate E/F for image {i}: {eng:.6f}")
            image.calc = None
            self.add_structure((image.copy(), eng, forces))
        self.fit()
        self.validate_data()
        self.set_K_inv()

    @classmethod
    def load_from_dict(cls, dict0, device='cuda'):
        """Rebuild kernel, descriptor and noise settings from a saved dictionary (:1118-1161)."""
        instance = cls(kernel=None, descriptor=None, base_potential=None)
        if dict0["kernel"]["name"] in ["RBF", "RBF_mb"]:
            instance.kernel = RBF_mb()
        elif dict0["kernel"]["name"] in ["Dot", "Dot_mb"]:
            instance.kernel = Dot_mb()
        else:
            raise NotImplementedError("unknown kernel {:s}".format(dict0["kernel"]["name"]))
        instance.kernel.load_from_dict(dict0["kernel"])

        if dict0["descriptor"]["_type"] == "SO3":
            instance.descriptor = _lazy_SO3()()
            instance.descriptor.load_from_dict(dict0["descriptor"])
        else:
            raise NotImplementedError("unknown descriptors {:s}".format(str(dict0["descriptor"].get("name"))))

        from .device import MAX_DESCRIPTOR
        n_, l_ = instance.descriptor.nmax, instance.descriptor.lmax
        if n_ * (n_ + 1) // 2 * (l_ + 1) > MAX_DESCRIPTOR:      # before every descriptor of the database is recomputed
            raise NotImplementedError("SO3(nmax=%d, lmax=%d) gives descriptors of %d entries; the device kernels support %d"
                                      % (n_, l_, n_ * (n_ + 1) // 2 * (l_ + 1), MAX_DESCRIPTOR))
        if "base_potential" in dict0.keys():
            raise NotImplementedError("base potentials are outside the B200 hot path (SURVEY.md §2.1 #13)")
        instance.kernel.device = device
        instance.noise_e = dict0["noise"]["energy"]
        instance.noise_f = dict0["noise"]["force"]
        instance.f_coef = dict0["noise"]["f_coef"]
        instance.noise_bounds = dict0["noise"]["bounds"]
        return instance


ctypes_double = ctypes.c_double


def CUR_device(K, l_tol=1e-10):
    """CUR on a device-resident block: same selection as CUR() below (cuSOLVER syevd + leverage scores in
    gprb_cur_scores; the block is copied because the decomposition works in place)."""
    n = K.shape[0]
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    A = K.clone().contiguous()
    w = np.zeros(n)
    omega = torch.empty(n, dtype=F64, device="cuda")
    n_low = ctypes.c_int(0)
    _lib.call("gprb_cur_scores", ptr(A), A.stride(0), n, float(l_tol), w.ctypes.data, ptr(omega), ctypes.byref(n_low), stream())
    if n_low.value == 0:
        return np.zeros(0, dtype=np.int64)
    return np.argsort(-1 * omega.cpu().numpy(), kind="stable")[:n_low.value]


def CUR(K, l_tol=1e-10):
    """CUR selection of the rows most aligned with the near-null space of K
    (Jinnouchi et al., PRB 100, 014105 (2019), App. D; gaussianprocess.py:1165-1182)."""
    L, U = np.linalg.eigh(K)
    low = L < l_tol
    omega = (U[:, low] ** 2).sum(axis=1)
    ids = np.argsort(-1 * omega)
    return ids[:int(low.sum())]
