"""Device-side plumbing: packs (device-resident operands) and covariance assembly.

PyTorch is used only as the owner of device buffers and streams; every computation is a call
into libgpr_b200.so (include/gpr_b200.h).  There is no CPU fallback.
"""
import ctypes
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import c_vp, c_int

F64 = torch.float64
MAX_DESCRIPTOR = 64         # 16 k-steps of the DMMA kernels (csrc/cov_mma.cu)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("gpr_calculator_b200 needs an NVIDIA B200 (CUDA device); there is no CPU fallback")
    _lib.load()


def stream():
    return c_vp(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (or NULL)."""
    return c_vp(0) if t is None else c_vp(t.data_ptr())


def empty(*shape):
    return torch.empty(shape, dtype=F64, device="cuda")


class Pack:
    """Device-resident packed side of a covariance block (``gprb_pack``).

    x [R, d] float64, ele [R] int, indices = rows per group (the reference's packed tuple layout,
    utilities.py:340-390); dxdr [R, d, 3] makes it a force pack.  Arrays may be numpy (host) or
    torch CUDA tensors.
    """

    def __init__(self, x, ele, indices, dxdr=None, norm_eps=0.0):
        require_cuda()
        self.handle = c_vp(0)
        keep = []

        def as_ptr(a, dtype_np, dtype_t):
            if a is None:
                return c_vp(0)
            if isinstance(a, torch.Tensor):
                a = a.to(dtype=dtype_t).contiguous()
                keep.append(a)
                return c_vp(a.data_ptr())
            a = np.ascontiguousarray(a, dtype=dtype_np)
            keep.append(a)
            return c_vp(a.ctypes.data)

        rows = np.ascontiguousarray(np.asarray(indices, dtype=np.int64), dtype=np.int32)
        n_rows = int(rows.sum()) if len(rows) else 0
        if x is None or len(x) == 0:
            d = 1 if x is None or getattr(x, "ndim", 2) < 2 else int(x.shape[1])
        else:
            d = int(x.shape[1])
            if int(x.shape[0]) != n_rows:
                raise ValueError("sum(indices)=%d does not match the %d rows of x" % (n_rows, int(x.shape[0])))
            if int(len(ele)) != n_rows:
                raise ValueError("ele has %d entries for %d rows" % (len(ele), n_rows))
            if dxdr is not None and tuple(dxdr.shape) != (n_rows, d, 3):
                raise ValueError("dxdr must have shape (%d, %d, 3), got %s" % (n_rows, d, tuple(dxdr.shape)))
        if d > MAX_DESCRIPTOR:      # fail before the rows are packed, not at the first covariance build
            raise _lib.GprB200Error(_lib.ERR_UNSUPPORTED, "descriptor length %d > %d is not supported by the device kernels "
                                    "(e.g. SO3 needs nmax (nmax + 1) / 2 * (lmax + 1) <= %d)" % (d, MAX_DESCRIPTOR, MAX_DESCRIPTOR))
        self.ncols = 0 if dxdr is None else 3
        self.n_groups = len(rows)
        self.n_rows = n_rows
        self.d = d
        self.indices = [int(v) for v in rows]
        _lib.call("gprb_pack_create", ctypes.byref(self.handle), c_int(len(rows)),
                  c_vp(rows.ctypes.data) if len(rows) else c_vp(0), c_int(d), c_int(self.ncols),
                  as_ptr(x, np.float64, F64), as_ptr(dxdr, np.float64, F64), as_ptr(ele, np.int32, torch.int32),
                  float(norm_eps), stream())

    def pair_count(self, other, g0=0, g1=None):
        g1 = self.n_groups if g1 is None else g1
        return int(_lib.load().gprb_pack_pair_count(self.handle, g0, g1, other.handle))

    @property
    def n_out(self):
        """Rows this side contributes to a covariance matrix."""
        return self.n_groups * (3 if self.ncols else 1)

    def __del__(self):
        try:
            if self.handle:
                _lib.load().gprb_pack_destroy(self.handle)
                self.handle = c_vp(0)
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------
# conversion of the reference's data containers into packs, with a cache for the training set
# ------------------------------------------------------------------------------------------------
_CACHE = {}


def _root(a):
    while isinstance(getattr(a, "base", None), np.ndarray):
        a = a.base
    return a


def _cached(kind, arrays, indices, build):
    """Pack of a packed tuple of host arrays, built once per (kind, identity of EVERY array, group sizes).

    The key carries the pack kind (an array used as energy data and as force data gives two packs), address / shape /
    strides of all arrays and the group sizes; an entry lives as long as all its arrays do.  Arrays mutated IN PLACE are not
    detected (GP replaces its training arrays on every change, gaussianprocess.py:579-629); call clear_cache() after
    doing so."""
    if not all(isinstance(a, np.ndarray) for a in arrays) or arrays[0].size == 0:
        return build()
    key = (kind,) + tuple((a.__array_interface__["data"][0], a.shape, a.strides, a.dtype.str) for a in arrays) + \
        (tuple(int(v) for v in indices),)
    hit = _CACHE.get(key)
    if hit is not None and all(r() is not None for r in hit[0]):
        return hit[1]
    pack = build()
    for k in [k for k, v in _CACHE.items() if any(r() is None for r in v[0])]:
        del _CACHE[k]
    try:
        _CACHE[key] = ([weakref.ref(_root(a)) for a in arrays], pack)
    except TypeError:
        pass
    return pack


def clear_cache():
    _CACHE.clear()


def energy_pack(data):
    """`data`: packed tuple (X, ELE, indices) or list of (x, ele) (kee_C input, rbf_kernel.py:26-30)."""
    if data is None:
        return None
    if isinstance(data, Pack):
        return data
    if isinstance(data, tuple):
        X, ELE, indices = data
        if len(indices) == 0:
            return None
        return _cached("energy", (X, ELE), indices, lambda: Pack(X, ELE, indices))
    if len(data) == 0:
        return None
    from .utilities import list_to_tuple
    X, ELE, indices = list_to_tuple(list(data), mode="energy")
    return Pack(X, ELE, indices)


def force_pack(data, norm_eps=0.0):
    """`data`: packed tuple (X, dXdR, ELE, indices), or list / object ndarray of (x, dxdr, ele)."""
    if data is None:
        return None
    if isinstance(data, Pack):
        return data
    if isinstance(data, tuple):
        X, dXdR, ELE, indices = data
        if len(indices) == 0:
            return None
        build = lambda: Pack(X, ELE, indices, dxdr=dXdR[:, :, :3] if dXdR.shape[2] != 3 else dXdR, norm_eps=norm_eps)  # noqa: E731
        return build() if norm_eps else _cached("force", (X, dXdR, ELE), indices, build)
    if len(data) == 0:
        return None
    from .utilities import list_to_tuple
    X, dXdR, ELE, indices = list_to_tuple(list(data), stress=False)
    return Pack(X, ELE, indices, dxdr=dXdR, norm_eps=norm_eps)


def stress_packs(data):
    """Force data whose dxdr carries 9 columns (3 force + 6 Voigt stress columns, gaussianprocess.py:862-864)
    -> (force Pack, stress Pack of columns 3:6, stress Pack of columns 6:9).  The Voigt columns enter the
    algebra exactly like force columns (rbf_kernel.cpp:642-822), so each triple is packed as a force side."""
    if isinstance(data, tuple) and len(data) == 3 and all(isinstance(p, Pack) for p in data):
        return data                                   # already split
    if not isinstance(data, tuple):
        from .utilities import list_to_tuple
        data = list_to_tuple(list(data), stress=True)
    X, dXdR, ELE, indices = data
    if dXdR.shape[2] != 9:
        raise ValueError("stress data needs dxdr with 9 columns, got %d" % dXdR.shape[2])
    cols = lambda a, b: dXdR[:, :, a:b] if isinstance(dXdR, torch.Tensor) else np.ascontiguousarray(dXdR[:, :, a:b])  # noqa: E731
    return tuple(Pack(X, ELE, indices, dxdr=cols(a, a + 3)) for a in (0, 3, 6))


def interleave_stress(Ka, Kb, n_groups):
    """[3 G, n] rows of the two stress triples -> [6 G, n] with rows (group, voigt 0..5)."""
    n = Ka.shape[1]
    return torch.cat((Ka.reshape(n_groups, 3, n), Kb.reshape(n_groups, 3, n)), dim=1).reshape(6 * n_groups, n)


def k_total_stress_device(kernel, p0, p1, zeta, data1, data2, use_tol=True, tol=1e-10, zeta_ef=None, zeta_ff=None):
    """(K [NE1 + 3 NF1, N2], K1 [6 NF1, N2]) between a test side whose force data carry the stress columns and a
    training side (k_total_with_stress, RBF_mb.py:206-229 / Dot_mb.py:150-173)."""
    require_cuda()
    e1 = energy_pack(data1["energy"]) if "energy" in data1 else None
    f1 = sa = sb = None
    if "force" in data1 and len(data1["force"]) > 0:
        f1, sa, sb = stress_packs(data1["force"])
    side2 = packs_of(data2)
    K, _ = k_total_device(kernel, p0, p1, zeta, (e1, f1), side2, use_tol=use_tol, tol=tol, grad=False,
                          zeta_ef=zeta_ef, zeta_ff=zeta_ff)
    if f1 is None:
        return K, None
    NF1, n_cols = f1.n_groups, K.shape[1]
    parts = []
    for spack in (sa, sb):
        Ks = torch.empty((3 * NF1, n_cols), dtype=F64, device="cuda")
        build_force_rows(kernel, p0, p1, zeta, (None, spack), side2, (0, NF1), Ks, None, use_tol=use_tol, tol=tol,
                         zeta_ef=zeta_ef, zeta_ff=zeta_ff, ff_mode=_lib.FF_FULL)
        parts.append(Ks)
    return K, interleave_stress(parts[0], parts[1], NF1)


def virial_packs(data, norm_eps=0.0):
    """Stress tuple of batch.virial_rows_from_batch (X, V [A, d, 6], ELE, indices) -> (force Pack of Voigt columns 0:3,
    force Pack of columns 3:6): the total-stress counterpart of the two stress triples of stress_packs."""
    X, V, ELE, indices = data
    return tuple(Pack(X, ELE, indices, dxdr=V[:, :, a:a + 3], norm_eps=norm_eps) for a in (0, 3))


def k_virial_device(kernel, p0, p1, zeta, packs, train_side, use_tol=True, tol=1e-10, zeta_ef=None, zeta_ff=None,
                    prior_packs=None, prior_tol=1e-12):
    """(K* [6 S, N2] with rows (structure, voigt 0..5), prior variance [6 S]) of the total stress of S structures.

    packs: virial_packs of the structures; train_side: (energy Pack, force Pack).  K* takes the K_fe / K_ff arguments of
    k_total_stress_device, so every row is the sum over atoms of that route's per-atom stress rows.  The prior is the
    FF_DIAG of each triple with diag_device's conventions: prior_packs (default `packs`; the Dot kernel passes packs with
    its norm_eps), `zeta` and prior_tol."""
    require_cuda()
    S = packs[0].n_groups
    NE2, NF2 = _sizes(train_side)
    n_cols = NE2 + 3 * NF2
    parts, prior = [], []
    for p, q in zip(packs, prior_packs or packs):
        Ks = torch.empty((3 * S, n_cols), dtype=F64, device="cuda")
        build_force_rows(kernel, p0, p1, zeta, (None, p), train_side, (0, S), Ks, None, use_tol=use_tol, tol=tol,
                         zeta_ef=zeta_ef, zeta_ff=zeta_ff, ff_mode=_lib.FF_FULL)
        parts.append(Ks)
        prior.append(diag_device(kernel, p0, p1, zeta, (None, q), tol=prior_tol).reshape(-1, 1))
    return interleave_stress(parts[0], parts[1], S), interleave_stress(prior[0], prior[1], S).reshape(-1)


def packs_of(data):
    """dict {'energy':…, 'force':…} -> (energy Pack or None, force Pack or None)."""
    e = energy_pack(data["energy"]) if "energy" in data else None
    f = force_pack(data["force"]) if "force" in data else None
    return e, f


# ------------------------------------------------------------------------------------------------
# covariance assembly  [[K_ee, K_ef], [K_fe, K_ff]]  (kernels/base.py:3-30 build_covariance)
# ------------------------------------------------------------------------------------------------
def _sizes(side):
    e, f = side
    return (e.n_groups if e is not None else 0), (f.n_groups if f is not None else 0)


def _at(t, r, c):
    """Pointer to element (r, c) of a row-major 2-D tensor view (or NULL)."""
    return c_vp(0) if t is None else c_vp(t.data_ptr() + (r * t.stride(0) + c) * t.element_size())


def build_energy_rows(kernel, p0, p1, zeta, side1, side2, window, K, dK=None, zeta_ef=None, kfe_rows=None, skip_kef=False):
    """Rows of side-1 energy groups [ea, eb): K[:, :NE2] = K_ee, K[:, NE2:] = K_ef.

    K / dK: [eb - ea, NE2 + 3 NF2] row-major views (a row stride > n_cols is fine).  When `kfe_rows`
    = (Kfe, dKfe) is given (training matrix, full window) the transposed block K_fe is written in
    the same pass ([3 NF, >= NE] views)."""
    e1, _ = side1
    e2, f2 = side2
    NE2, NF2 = _sizes(side2)
    ea, eb = window
    if e1 is None or eb <= ea:
        return
    zeta_ef = zeta if zeta_ef is None else zeta_ef
    st = stream()
    ld = K.stride(0)
    ldd = dK.stride(0) if dK is not None else 0
    if e2 is not None:
        _lib.call("gprb_kee", kernel, e1.handle, e2.handle, p0, p1, float(zeta), ea, eb, _at(K, 0, 0), ld, _at(dK, 0, 0), ldd, st)
    if f2 is None or skip_kef:
        return
    Kfe, dKfe = kfe_rows if kfe_rows is not None else (None, None)
    if (ea, eb) == (0, e1.n_groups):
        _lib.call("gprb_kef", kernel, e1.handle, f2.handle, p0, p1, float(zeta_ef), 0, NF2,
                  _at(K, 0, NE2), ld, _at(Kfe, 0, 0), Kfe.stride(0) if Kfe is not None else 0,
                  _at(dK, 0, NE2), ldd, _at(dKfe, 0, 0), dKfe.stride(0) if dKfe is not None else 0, st)
    else:
        # the K_ef kernel windows over force groups: build the full-height block, keep my rows
        tmp = torch.empty((e1.n_groups, 3 * NF2), dtype=F64, device="cuda")
        dtmp = torch.empty((e1.n_groups, 3 * NF2), dtype=F64, device="cuda") if dK is not None else None
        _lib.call("gprb_kef", kernel, e1.handle, f2.handle, p0, p1, float(zeta_ef), 0, NF2,
                  ptr(tmp), 3 * NF2, c_vp(0), 0, ptr(dtmp), 3 * NF2, c_vp(0), 0, st)
        K[:, NE2:NE2 + 3 * NF2] = tmp[ea:eb]
        if dK is not None:
            dK[:, NE2:NE2 + 3 * NF2] = dtmp[ea:eb]


def build_force_rows(kernel, p0, p1, zeta, side1, side2, window, K, dK=None, use_tol=True, tol=1e-10,
                     zeta_ef=None, zeta_ff=None, ff_mode=_lib.FF_FULL, skip_kfe=False, peer_slabs=None):
    """Rows of side-1 force groups [fa, fb): K[:, :NE2] = K_fe, K[:, NE2:] = K_ff.

    K / dK: [3 (fb - fa), NE2 + 3 NF2] row-major views.  ff_mode: FF_FULL, FF_SYMMETRIC (side1 is
    side2, full window, mirrored entries written) or FF_UPPER (side1 is side2: only blocks J >= I
    are written; finish with gprb_symmetrize).
    peer_slabs: device addresses of the same row slab (element (0, 0) of `K`) in the other ranks' copies of
    the matrix (dist.PeerMatrix): the kernels store every finished value into all copies (fused gather,
    gprb_kff_multi / gprb_kfe_multi); K is then NOT zeroed by the call, the caller has zeroed every copy."""
    _, f1 = side1
    e2, f2 = side2
    NE2, NF2 = _sizes(side2)
    fa, fb = window
    if f1 is None or fb <= fa:
        return
    zeta_ef = zeta if zeta_ef is None else zeta_ef
    zeta_ff = zeta if zeta_ff is None else zeta_ff
    st = stream()
    ld = K.stride(0)
    ldd = dK.stride(0) if dK is not None else 0
    if peer_slabs:
        n_dst = 1 + len(peer_slabs)
        if n_dst > _lib.MAX_DST:
            raise ValueError("at most %d destination matrices" % _lib.MAX_DST)
        base = K.data_ptr()
        if e2 is not None and not skip_kfe:
            dst = (c_vp * n_dst)(base, *[int(q) for q in peer_slabs])
            _lib.call("gprb_kfe_multi", kernel, e2.handle, f1.handle, p0, p1, float(zeta_ef), fa, fb,
                      n_dst, dst, ld, _at(dK, 0, 0), ldd, st)
        if f2 is not None:
            dst = (c_vp * n_dst)(base + NE2 * 8, *[int(q) + NE2 * 8 for q in peer_slabs])
            _lib.call("gprb_kff_multi", kernel, f1.handle, f2.handle, p0, p1, float(zeta_ff), int(bool(use_tol)), float(tol),
                      ff_mode, fa, fb, n_dst, dst, ld, _at(dK, 0, NE2), ldd, st)
        return
    if e2 is not None and not skip_kfe:
        _lib.call("gprb_kef", kernel, e2.handle, f1.handle, p0, p1, float(zeta_ef), fa, fb,
                  c_vp(0), 0, _at(K, 0, 0), ld, c_vp(0), 0, _at(dK, 0, 0), ldd, st)
    if f2 is not None:
        _lib.call("gprb_kff", kernel, f1.handle, f2.handle, p0, p1, float(zeta_ff), int(bool(use_tol)), float(tol),
                  ff_mode, fa, fb, _at(K, 0, NE2), ld, _at(dK, 0, NE2), ldd, st)


def k_total_device(kernel, p0, p1, zeta, side1, side2=None, use_tol=True, tol=1e-10, grad=False,
                   zeta_ef=None, zeta_ff=None, window=None, symmetric=True):
    """Build the covariance between two (energy Pack, force Pack) sides on the current CUDA device.

    window = ((e0, e1), (f0, f1)): only the rows of side-1 energy groups [e0,e1) and force groups
    [f0,f1) are computed (row-block sharding).  Returns (K, dK) torch tensors of shape
    [rows, NE2 + 3 NF2]; dK is dK/dl for RBF when grad=True, else None.
    """
    require_cuda()
    same = side2 is None
    side2 = side1 if same else side2
    NE1, NF1 = _sizes(side1)
    NE2, NF2 = _sizes(side2)
    if window is None:
        (ea, eb), (fa, fb) = (0, NE1), (0, NF1)
    else:
        (ea, eb), (fa, fb) = window
    full = (ea, eb, fa, fb) == (0, NE1, 0, NF1)
    n_rows = (eb - ea) + 3 * (fb - fa)
    n_cols = NE2 + 3 * NF2
    # every block that exists for the given sides is fully written by its builder
    K = torch.empty((n_rows, n_cols), dtype=F64, device="cuda")
    dK = torch.empty((n_rows, n_cols), dtype=F64, device="cuda") if grad else None
    if n_rows == 0 or n_cols == 0:
        return K, dK
    r_f = eb - ea          # first force row of the block
    one_pass = same and full and side1[0] is not None and side1[1] is not None
    build_energy_rows(kernel, p0, p1, zeta, side1, side2, (ea, eb), K[:r_f], None if dK is None else dK[:r_f],
                      zeta_ef=zeta_ef, kfe_rows=(K[r_f:], None if dK is None else dK[r_f:]) if one_pass else None)
    mode = _lib.FF_SYMMETRIC if (same and full and symmetric) else _lib.FF_FULL
    build_force_rows(kernel, p0, p1, zeta, side1, side2, (fa, fb), K[r_f:], None if dK is None else dK[r_f:],
                     use_tol=use_tol, tol=tol, zeta_ef=zeta_ef, zeta_ff=zeta_ff, ff_mode=mode, skip_kfe=one_pass)
    return K, dK


def diag_device(kernel, p0, p1, zeta, side, tol=1e-12):
    """Prior variance of every row of `side` (RBF_mb.diag, RBF_mb.py:62-133; Dot_mb.diag)."""
    require_cuda()
    e, f = side
    NE = e.n_groups if e is not None else 0
    NF = f.n_groups if f is not None else 0
    out = torch.zeros(NE + 3 * NF, dtype=F64, device="cuda")
    st = stream()
    if e is not None:
        _lib.call("gprb_kee_diag", kernel, e.handle, p0, p1, float(zeta), ptr(out), st)
    if f is not None:
        _lib.call("gprb_kff", kernel, f.handle, f.handle, p0, p1, float(zeta), 1, float(tol), _lib.FF_DIAG, 0, NF,
                  c_vp(out.data_ptr() + NE * 8), 0, c_vp(0), 0, st)
    return out
