"""GPU: the factored K_ff + dK/dl build (csrc/cov_factored.cu) against the pairwise kernel (GPRB_KFF_FACTORED=0) on
the same packs: S5-like Cu32 packs in FULL, SYMMETRIC and UPPER mode, Pd4/MgO structures with three species (clusters
cut inside a 220-atom structure) and 108-atom structures.  Per entry K within 1e-12 of sqrt(K_ii K_jj), dK/dl within
1e-12 of that scale times (1/l^3 + 2/l), every entry within 1e-13 of the block's largest; UPPER leaves the blocks below
the diagonal zero; two builds are bitwise equal."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
SIGMA, ELL, ZETA = 1.0, 0.1, 2.0


def _des():
    from gpr_calculator_b200.SO3 import SO3
    return SO3(nmax=3, lmax=4, rcut=5.0)


def _pack(atoms_list):
    from gpr_calculator_b200 import device as gdev, synthetic as syn
    _, F = syn.packed_from_batch(_des(), atoms_list)
    return gdev.Pack(F[0], F[2], F[3], dxdr=F[1])


def _build(f, mode, factored, sigma=SIGMA, ell=ELL, zeta=ZETA):
    """K, dK/dl and the number of kernels launched; factored: None (cost model), '0' or '1' (GPRB_KFF_FACTORED)."""
    from gpr_calculator_b200 import _lib, device as gdev
    NF = f.n_groups
    K = torch.full((3 * NF, 3 * NF), float("nan"), dtype=torch.float64, device="cuda")
    dK = torch.full((3 * NF, 3 * NF), float("nan"), dtype=torch.float64, device="cuda")
    old = os.environ.pop("GPRB_KFF_FACTORED", None)
    if factored is not None:
        os.environ["GPRB_KFF_FACTORED"] = factored
    try:
        n0 = _lib.load().gprb_launch_count()
        _lib.call("gprb_kff", _lib.RBF, f.handle, f.handle, sigma, ell, zeta, 0, 1e-10, mode, 0, NF,
                  gdev.ptr(K), 3 * NF, gdev.ptr(dK), 3 * NF, gdev.stream())
        torch.cuda.synchronize()
        n = _lib.load().gprb_launch_count() - n0
    finally:
        os.environ.pop("GPRB_KFF_FACTORED", None)
        if old is not None:
            os.environ["GPRB_KFF_FACTORED"] = old
    return K, dK, n


def _check(Kf, dKf, Kp, dKp, ell=ELL, min_var=0.0):
    """Per entry on the Cauchy-Schwarz scale sqrt(K_ii K_jj) (dK/dl: times 1/l^3 + 2/l) over the rows whose prior variance
    K_ii is at least min_var of the largest, and every entry within 1e-13 of the block's largest |K| / |dK/dl|."""
    assert torch.isfinite(Kf).all() and torch.isfinite(dKf).all()
    diag = torch.diagonal(Kp)
    keep = diag >= min_var * diag.max()
    d = torch.sqrt(torch.clamp(diag[keep], min=0))
    scale = torch.outer(d, d) + 1e-300
    sub = lambda M: M[keep][:, keep]
    errK = float((sub(Kf - Kp).abs() / scale).max())
    errdK = float((sub(dKf - dKp).abs() / (scale * (1 / ell ** 3 + 2 / ell))).max())
    assert errK <= 1e-12, errK
    assert errdK <= 1e-12, errdK
    assert float((Kf - Kp).abs().max()) <= 1e-13 * float(Kp.abs().max())
    assert float((dKf - dKp).abs().max()) <= 1e-13 * float(dKp.abs().max())


@pytest.fixture(scope="module")
def cu32():
    from gpr_calculator_b200 import synthetic as syn
    return _pack([a for a, _, _ in syn.structures(100, 2, 4000)])


@pytest.mark.parametrize("mode_name", ["FULL", "SYMMETRIC", "UPPER"])
def test_factored_matches_pairwise_cu32(cu32, mode_name):
    from gpr_calculator_b200 import _lib
    mode = getattr(_lib, "FF_" + mode_name)
    Kp, dKp, n_pair = _build(cu32, mode, "0")
    Kf, dKf, n_fact = _build(cu32, mode, None)          # the cost model picks the factored build at this shape
    assert n_pair == 1 and n_fact >= 2
    if mode == _lib.FF_UPPER:
        # the diagonal of an UPPER build is complete; compare the written blocks, check the rest is zero
        NF = cu32.n_groups
        blk = torch.arange(3 * NF, device="cuda") // 3
        lower = blk[:, None] > blk[None, :]
        assert (Kf[lower] == 0).all() and (dKf[lower] == 0).all()
        assert (Kp[lower] == 0).all()
    _check(Kf, dKf, Kp, dKp)
    Kf2, dKf2, _ = _build(cu32, mode, None)
    assert torch.equal(Kf, Kf2) and torch.equal(dKf, dKf2)


def test_factored_matches_pairwise_pd4_three_species():
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.utilities import SimpleAtoms
    g = np.load(os.path.join(GOLD, "pd4.npz"))
    atoms = [SimpleAtoms(list(g["numbers"]), g["positions"][k], g["cell"], pbc=g["pbc"]) for k in (0, 50, 100)]
    f = _pack(atoms)
    assert len(set(g["numbers"].tolist())) == 3
    for zeta, ell in ((2.0, 0.7), (3.0, 0.4)):
        Kp, dKp, _ = _build(f, _lib.FF_UPPER, "0", ell=ell, zeta=zeta)
        Kf, dKf, n = _build(f, _lib.FF_UPPER, "1", ell=ell, zeta=zeta)
        assert n >= 2
        # atoms at symmetric sites of the MgO slab have force variances that are sums cancelling to ~1e-11 of the
        # largest: on their own scale the last-bit differences of a reordered sum are not meaningful (rows down to
        # 1e-6 of the largest variance: 1.2e-11 per entry, an absolute difference of ~1e-17 of the largest entry)
        _check(Kf, dKf, Kp, dKp, ell=ell, min_var=1e-2)


def test_factored_matches_pairwise_cu108():
    from gpr_calculator_b200 import _lib, synthetic as syn
    f = _pack([a for a, _, _ in syn.structures(4, 3, 5000)])
    for mode in (_lib.FF_UPPER, _lib.FF_FULL):
        Kp, dKp, _ = _build(f, mode, "0")
        Kf, dKf, n = _build(f, mode, "1")
        assert n >= 2
        _check(Kf, dKf, Kp, dKp)
