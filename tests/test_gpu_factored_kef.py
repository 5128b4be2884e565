"""GPU: the factored K_fe / K_ef + dK/dl build (csrc/cov_factored.cu) against the pairwise kernel (GPRB_KFF_FACTORED=0)
on the packs of test_gpu_factored_kff.py: S5-like Cu32 structures, Pd4/MgO structures with three species and 108-atom
structures.  Per entry within 1e-12 of sqrt(K_ee[I,I] K_ff[3J+c,3J+c]) (dK/dl: times 1/l^3 + 2/l), every entry within
1e-13 of the block's largest, K_ef == K_fe^T bit for bit, and two builds bitwise equal."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
SIGMA, ELL, ZETA = 1.0, 0.1, 2.0


def _packs(atoms_list):
    from gpr_calculator_b200 import device as gdev, synthetic as syn
    from gpr_calculator_b200.SO3 import SO3
    E, F = syn.packed_from_batch(SO3(nmax=3, lmax=4, rcut=5.0), atoms_list)
    return gdev.Pack(E[0], E[1], E[2]), gdev.Pack(F[0], F[2], F[3], dxdr=F[1])


def _with_switch(factored, fn):
    old = os.environ.pop("GPRB_KFF_FACTORED", None)
    if factored is not None:
        os.environ["GPRB_KFF_FACTORED"] = factored
    try:
        return fn()
    finally:
        os.environ.pop("GPRB_KFF_FACTORED", None)
        if old is not None:
            os.environ["GPRB_KFF_FACTORED"] = old


def _build(e, f, factored, sigma=SIGMA, ell=ELL, zeta=ZETA, fe=True):
    """K_ef, K_fe, dK_ef/dl, dK_fe/dl and the number of kernels launched; factored: None (cost model), '0' or '1'.
    fe=False: the K_ef outputs only (K_fe and dK_fe/dl NULL)."""
    from gpr_calculator_b200 import _lib, device as gdev
    NE, NF = e.n_groups, f.n_groups
    new = lambda r, c: torch.full((r, c), float("nan"), dtype=torch.float64, device="cuda")
    Kef, dKef = new(NE, 3 * NF), new(NE, 3 * NF)
    Kfe, dKfe = (new(3 * NF, NE), new(3 * NF, NE)) if fe else (None, None)

    def run():
        n0 = _lib.load().gprb_launch_count()
        _lib.call("gprb_kef", _lib.RBF, e.handle, f.handle, sigma, ell, zeta, 0, NF,
                  gdev.ptr(Kef), 3 * NF, gdev.ptr(Kfe), NE, gdev.ptr(dKef), 3 * NF, gdev.ptr(dKfe), NE, gdev.stream())
        torch.cuda.synchronize()
        return _lib.load().gprb_launch_count() - n0
    n = _with_switch(factored, run)
    return Kef, Kfe, dKef, dKfe, n


def _diagonals(e, f, sigma, ell, zeta):
    """K_ee[I, I] and K_ff[3J+c, 3J+c] through the pairwise kernels."""
    from gpr_calculator_b200 import _lib, device as gdev
    NE, NF = e.n_groups, f.n_groups
    Kee = torch.empty((NE, NE), dtype=torch.float64, device="cuda")
    kff = torch.empty(3 * NF, dtype=torch.float64, device="cuda")
    _lib.call("gprb_kee", _lib.RBF, e.handle, e.handle, sigma, ell, zeta, 0, NE, gdev.ptr(Kee), NE, gdev.ptr(None), 0,
              gdev.stream())
    _lib.call("gprb_kff", _lib.RBF, f.handle, f.handle, sigma, ell, zeta, 0, 1e-10, _lib.FF_DIAG, 0, NF,
              gdev.ptr(kff), 0, gdev.ptr(None), 0, gdev.stream())
    torch.cuda.synchronize()
    return torch.diagonal(Kee).clone(), kff


def _check(got, ref, kee, kff, ell, min_var=0.0):
    Kef, _, dKef, _ = got[:4]
    Kp, _, dKp, _ = ref[:4]
    assert torch.isfinite(Kef).all() and torch.isfinite(dKef).all()
    ke, kf = kee >= min_var * kee.max(), kff >= min_var * kff.max()
    scale = torch.sqrt(torch.outer(torch.clamp(kee[ke], min=0), torch.clamp(kff[kf], min=0))) + 1e-300
    sub = lambda M: M[ke][:, kf]
    errK = float((sub(Kef - Kp).abs() / scale).max())
    errdK = float((sub(dKef - dKp).abs() / (scale * (1 / ell ** 3 + 2 / ell))).max())
    assert errK <= 1e-12, errK
    assert errdK <= 1e-12, errdK
    assert float((Kef - Kp).abs().max()) <= 1e-13 * float(Kp.abs().max())
    assert float((dKef - dKp).abs().max()) <= 1e-13 * float(dKp.abs().max())


def _transposed(b):
    Kef, Kfe, dKef, dKfe = b[:4]
    assert torch.equal(Kef, Kfe.T) and torch.equal(dKef, dKfe.T)


def test_factored_kef_matches_pairwise_cu32():
    from gpr_calculator_b200 import synthetic as syn
    e, f = _packs([a for a, _, _ in syn.structures(100, 2, 4000)])
    ref = _build(e, f, "0")
    got = _build(e, f, None)                   # the cost model picks the factored build at this shape
    assert ref[4] == 1 and got[4] >= 2
    _transposed(ref)
    _transposed(got)
    _check(got, ref, *_diagonals(e, f, SIGMA, ELL, ZETA), ell=ELL)
    again = _build(e, f, None)
    assert again[4] == 2                       # plan cached: the Y kernel and the contraction
    assert all(torch.equal(a, b) for a, b in zip(got[:4], again[:4]))
    only_ef = _build(e, f, None, fe=False)
    assert torch.equal(only_ef[0], got[0]) and torch.equal(only_ef[2], got[2])


def test_factored_kef_matches_pairwise_pd4_three_species():
    from gpr_calculator_b200.utilities import SimpleAtoms
    g = np.load(os.path.join(GOLD, "pd4.npz"))
    atoms = [SimpleAtoms(list(g["numbers"]), g["positions"][k], g["cell"], pbc=g["pbc"]) for k in (0, 50, 100)]
    e, f = _packs(atoms)
    for zeta, ell in ((2.0, 0.7), (3.0, 0.4)):
        ref = _build(e, f, "0", ell=ell, zeta=zeta)
        got = _build(e, f, "1", ell=ell, zeta=zeta)
        assert ref[4] == 1 and got[4] >= 2
        _transposed(got)
        # force rows of atoms at symmetric sites of the MgO slab have variances that cancel to ~1e-11 of the largest:
        # the per-entry bound is taken over rows down to 1e-2 of the largest variance, as for K_ff
        _check(got, ref, *_diagonals(e, f, SIGMA, ell, zeta), ell=ell, min_var=1e-2)


def test_factored_kef_matches_pairwise_cu108():
    from gpr_calculator_b200 import synthetic as syn
    e, f = _packs([a for a, _, _ in syn.structures(4, 3, 5000)])
    ref = _build(e, f, "0")
    got = _build(e, f, "1")
    assert ref[4] == 1 and got[4] >= 2
    _transposed(got)
    _check(got, ref, *_diagonals(e, f, SIGMA, ELL, ZETA), ell=ELL)
