"""GPU parity: covariance blocks of libgpr_b200 (through the C-ABI, via the reference-shaped wrappers)
against the golden vectors of the reference and the CPU oracle.  Tolerance from north_star:
K entries within 1e-10 relative (of the block's largest entry: entries that are sums of cancelling
terms are compared on the block scale, SURVEY.md §7.3)."""
import os

import numpy as np
import pytest
import torch

from helpers import make_force, make_energy, rel_err, entry_err

pytestmark = pytest.mark.gpu
TOL = 1e-10
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gk():
    return np.load(os.path.join(GOLD, "kernels.npz"))


def _inputs(g):
    F1 = (g["F1_x"], g["F1_dxdr"], g["F1_ele"], list(g["F1_ind"]))
    F2 = (g["F2_x"], g["F2_dxdr"], g["F2_ele"], list(g["F2_ind"]))
    E1 = (g["E1_x"], g["E1_ele"], list(g["E1_ind"]))
    E2 = (g["E2_x"], g["E2_ele"], list(g["E2_ind"]))
    return E1, E2, F1, F2


def test_library_loaded_and_device_is_blackwell():
    from gpr_calculator_b200 import _lib
    import ctypes
    sm, maj, mnr = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.call("gprb_device_info", ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr))
    assert sm.value > 0 and maj.value >= 10


def test_rbf_blocks_vs_golden(gk):
    from gpr_calculator_b200.kernels import rbf_kernel as rk
    E1, E2, F1, F2 = _inputs(gk)
    sig, l = gk["params"]
    for zeta in (2.0, 3.0):
        z = "z%d" % int(zeta)
        assert rel_err(rk.kee_C(E1, E2, sig, l, zeta), gk["rbf_kee_" + z]) <= TOL
        assert rel_err(rk.kef_C(E1, F2, sig, l, zeta), gk["rbf_kef_" + z]) <= TOL
        assert rel_err(rk.kff_C(F1, F2, sig, l, zeta, tol=1e-12), gk["rbf_kff_" + z]) <= TOL
        for name, fn, a, b in (("kee", rk.kee_C, E1, E2), ("kef", rk.kef_C, E1, F2), ("kff", rk.kff_C, F1, F2)):
            for k, v in zip(("K", "Ks", "Kl"), fn(a, b, sig, l, zeta, grad=True)):
                assert rel_err(v, gk["rbf_%s_grad_%s_%s" % (name, k, z)]) <= TOL, (name, k, z)
    # the pair cut `dK_dD > tol` (rbf_kernel.cpp:395) with a tol that really removes pairs
    assert rel_err(rk.kff_C(F1, F2, 1.0, 0.2, 2.0, tol=1.0), gk["rbf_kff_tol_l02"]) <= TOL
    assert rel_err(rk.kef_C(E1, F2, sig, l, 2.0, transpose=True), gk["rbf_kef_z2"].T) <= TOL


def test_dot_blocks_vs_golden(gk):
    from gpr_calculator_b200.kernels import dot_kernel as dk
    E1, E2, F1, F2 = _inputs(gk)
    for zeta in (2.0, 3.0):
        z = "z%d" % int(zeta)
        assert rel_err(dk.kee_C(E1, E2, 2.0, 1.5, zeta), gk["dot_kee_" + z]) <= TOL
        assert rel_err(dk.kef_C(E1, F2, 2.0, 1.5, zeta), gk["dot_kef_" + z]) <= TOL
        assert rel_err(dk.kff_C(F1, F2, 2.0, 1.5, zeta), gk["dot_kff_" + z]) <= TOL


def test_kernel_objects_vs_golden(gk):
    """RBF_mb / Dot_mb assembled matrices incl. the reference quirks (Dot zeta slot, eps diag)."""
    from gpr_calculator_b200.kernels import RBF_mb, Dot_mb
    from gpr_calculator_b200.utilities import tuple_to_list
    E1, E2, F1, F2 = _inputs(gk)
    sig, l = gk["params"]
    data, data2 = {"energy": E1, "force": F1}, {"energy": E2, "force": F2}
    rbf = RBF_mb(para=[sig, l], zeta=2)
    K = rbf.k_total(data)
    assert rel_err(K, gk["RBF_k_total"]) <= TOL
    assert np.abs(K - K.T).max() <= 1e-12 * np.abs(K).max()
    assert rel_err(rbf.k_total(data2, data, f_tol=1e-12), gk["RBF_k_total_rect"]) <= TOL
    K, dK = rbf.k_total_with_grad(data)
    assert rel_err(K, gk["RBF_k_grad_K"]) <= TOL and rel_err(dK, gk["RBF_k_grad_dK"]) <= TOL
    assert rel_err(rbf.diag({"energy": E1, "force": tuple_to_list(F1)}), gk["RBF_diag"]) <= TOL
    dot = Dot_mb(para=[2.0, 1.5], zeta=3)
    assert rel_err(dot.k_total(data), gk["Dot_k_total"]) <= TOL
    K, dK = dot.k_total_with_grad(data)
    assert rel_err(K, gk["Dot_k_grad_K"]) <= TOL and rel_err(dK, gk["Dot_k_grad_dK"]) <= TOL
    assert rel_err(dot.diag({"energy": tuple_to_list(E1, mode="energy"), "force": tuple_to_list(F1)}), gk["Dot_diag"]) <= 1e-9
    with pytest.raises(ValueError):
        dot.diag({"force": F1})      # packed tuple rejected like Dot_mb.py:71-78


CASES = [
    # (name, kwargs for make_force side 1, side 2)
    ("ragged", dict(n_groups=9, lo=3, hi=40), dict(n_groups=7, lo=3, hi=40)),
    ("single_rows", dict(n_groups=13, lo=1, hi=2), dict(n_groups=5, lo=1, hi=9)),
    ("large_split_groups", dict(n_groups=3, lo=70, hi=150), dict(n_groups=4, lo=60, hi=100)),
    ("zero_norm_rows", dict(n_groups=6, lo=4, hi=12, zero_rows=2), dict(n_groups=6, lo=4, hi=12, zero_rows=1)),
    ("three_species", dict(n_groups=6, lo=5, hi=30, species=(1, 16, 46)), dict(n_groups=5, lo=5, hi=30, species=(1, 16, 46))),
    ("d24", dict(n_groups=5, lo=5, hi=20, d=24), dict(n_groups=4, lo=5, hi=20, d=24)),
    ("d7", dict(n_groups=5, lo=5, hi=20, d=7), dict(n_groups=4, lo=5, hi=20, d=7)),
    ("d32", dict(n_groups=4, lo=5, hi=20, d=32), dict(n_groups=4, lo=5, hi=20, d=32)),
    ("big_norms", dict(n_groups=5, lo=20, hi=35, scale=7e3), dict(n_groups=5, lo=20, hi=35, scale=7e3)),
    # descriptors of 33..64 entries (e.g. SO3(nmax=4, lmax=4): d = 50) take the 6-warp / 16-k-step instantiations
    ("d40", dict(n_groups=7, lo=5, hi=30, d=40), dict(n_groups=5, lo=5, hi=30, d=40)),
    ("d50", dict(n_groups=9, lo=3, hi=60, d=50, species=(1, 16, 46)), dict(n_groups=6, lo=3, hi=60, d=50, species=(1, 16, 46))),
    ("d64", dict(n_groups=4, lo=40, hi=70, d=64), dict(n_groups=5, lo=1, hi=20, d=64)),
]


@pytest.mark.parametrize("name,kw1,kw2", CASES, ids=[c[0] for c in CASES])
def test_blocks_vs_oracle(oracle_libs, name, kw1, kw2):
    """Seeded ragged inputs, edge cases of the domain (single-row groups, groups split over CTAs,
    dropped zero-norm rows, species masks, descriptor lengths) against the CPU oracle."""
    from gpr_calculator_b200.kernels import rbf_kernel as rk, dot_kernel as dk
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(1000 + [c[0] for c in CASES].index(name))      # deterministic per case
    d = kw1.get("d", 30)
    F1, F2 = list_to_tuple(make_force(rng, **kw1)), list_to_tuple(make_force(rng, **kw2))
    ekw = dict(d=d, species=kw1.get("species", (13, 79)), scale=kw1.get("scale", 1.0))
    E1 = list_to_tuple(make_energy(rng, 4, **ekw), mode="energy")
    E2 = list_to_tuple(make_energy(rng, 3, lo=1, hi=130, **ekw), mode="energy")
    O, OD = oracle_libs.RBFOracle("port"), oracle_libs.DotOracle("port")
    sig, l = 1.7, 0.6
    for zeta in (2.0, 3.0, 2.5):
        # prior variances of every row of the four sides: the per-entry (Cauchy-Schwarz) scale, helpers.entry_err
        dF1, dF2 = np.diag(O.kff_C(F1, F1, sig, l, zeta, tol=0.0)), np.diag(O.kff_C(F2, F2, sig, l, zeta, tol=0.0))
        dE1, dE2 = np.diag(O.kee_C(E1, E1, sig, l, zeta)), np.diag(O.kee_C(E2, E2, sig, l, zeta))
        hl = 1.0 / l ** 3 + 2.0 / l          # bound of |d log k / dl|: scale of the dK/dl entries
        for grad in (False, True):
            for fn_g, fn_o, a, b, da, db in ((rk.kff_C, O.kff_C, F1, F2, dF1, dF2), (rk.kef_C, O.kef_C, E1, F2, dE1, dF2),
                                             (rk.kee_C, O.kee_C, E1, E2, dE1, dE2)):
                got, ref = fn_g(a, b, sig, l, zeta, grad=grad), fn_o(a, b, sig, l, zeta, grad=grad)
                got, ref = (got, ref) if grad else ((got,), (ref,))
                for k, (x, y) in enumerate(zip(got, ref)):
                    assert x.shape == y.shape and rel_err(x, y) <= TOL, (name, zeta, grad, fn_g.__name__)
                    s_k = (1.0, 2.0 / sig, hl)[k]        # K, dK/dsigma = 2K/sigma, dK/dl
                    assert entry_err(x, y, da * s_k, db * s_k) <= TOL, (name, zeta, grad, fn_g.__name__, "per entry", k)
        assert rel_err(dk.kff_C(F1, F2, 2.0, 1.5, zeta), OD.kff_C(F1, F2, 2.0, 1.5, zeta)) <= TOL
        assert rel_err(dk.kef_C(E1, F2, 2.0, 1.5, zeta), OD.kef_C(E1, F2, 2.0, 1.5, zeta)) <= TOL
        assert rel_err(dk.kee_C(E1, E2, 2.0, 1.5, zeta), OD.kee_C(E1, E2, 2.0, 1.5, zeta)) <= TOL


def test_disjoint_species_give_zero():
    from gpr_calculator_b200.kernels import rbf_kernel as rk
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(5)
    F1 = list_to_tuple(make_force(rng, 3, species=(13,)))
    F2 = list_to_tuple(make_force(rng, 4, species=(79,)))
    assert np.count_nonzero(rk.kff_C(F1, F2, 1.0, 0.5, 2.0)) == 0


def test_descriptor_longer_than_64_fails_loudly():
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.kernels import rbf_kernel as rk
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(6)
    F = list_to_tuple(make_force(rng, 2, d=72))
    with pytest.raises(_lib.GprB200Error):
        rk.kff_C(F, F, 1.0, 0.5, 2.0)


def test_modes_and_windows_agree():
    """Symmetric build == full build; row windows concatenate to the full matrix; diag mode ==
    diagonal of the block; K(sigma) = sigma^2 K(1) (size-independent properties)."""
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import Pack, k_total_device, diag_device
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(7)
    X, dX, ELE, ind = list_to_tuple(make_force(rng, 41, lo=20, hi=36))
    Xe, Ee, inde = list_to_tuple(make_energy(rng, 9, lo=20, hi=40), mode="energy")
    f, e = Pack(X, ELE, ind, dxdr=dX), Pack(Xe, Ee, inde)
    for kern, p1 in ((_lib.RBF, 0.7), (_lib.DOT, 1.1)):
        grad = kern == _lib.RBF
        Ks, dKs = k_total_device(kern, 1.3, p1, 2.0, (e, f), None, use_tol=False, grad=grad, symmetric=True)
        Kf, dKf = k_total_device(kern, 1.3, p1, 2.0, (e, f), None, use_tol=False, grad=grad, symmetric=False)
        scale = Kf.abs().max().item()
        assert (Ks - Kf).abs().max().item() <= 1e-13 * scale
        assert (Ks - Ks.T).abs().max().item() <= 1e-13 * scale
        if grad:
            assert (dKs - dKf).abs().max().item() <= 1e-13 * dKf.abs().max().item()
        rows = []
        for w in (((0, 4), (0, 13)), ((4, 9), (13, 41))):
            Kw, _ = k_total_device(kern, 1.3, p1, 2.0, (e, f), None, use_tol=False, grad=False, window=w)
            rows.append(Kw)
        NE = 9
        K2 = torch.cat((rows[0][:4], rows[1][:5], rows[0][4:], rows[1][5:]))
        assert (K2 - Kf).abs().max().item() <= 1e-13 * scale
        dg = diag_device(kern, 1.3, p1, 2.0, (None, f), tol=0.0)
        assert (dg - torch.diagonal(Kf)[NE:]).abs().max().item() <= 1e-13 * scale
        K1, _ = k_total_device(kern, 1.0, p1, 2.0, (e, f), None, use_tol=False, grad=False)
        assert (Kf - 1.3 ** 2 * K1).abs().max().item() <= 1e-13 * scale


def _lml_eval(K, dK_rows, ranges, NE, y, noise_e, noise_f):
    """gprb_lml_eval with the gradient traces on a copy of K (noise and factor are applied in place): out[0..5]."""
    import ctypes
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import ptr, stream
    N = K.shape[0]
    Kc = K.clone()
    alpha = torch.empty(N, dtype=torch.float64, device="cuda")
    n_work = int(_lib.load().gprb_lml_eval_work(N, NE, 1, 16))
    work = torch.empty(n_work, dtype=torch.float64, device="cuda")
    flat = [v for r in ranges for v in r]
    out = (ctypes.c_double * 8)()
    _lib.call("gprb_lml_eval", ptr(Kc), N, N, NE, ptr(y), float(noise_e), float(noise_f), ptr(dK_rows), dK_rows.stride(0),
              len(ranges), (ctypes.c_int * len(flat))(*flat), 1, 0, 16, 0, ptr(alpha), ptr(work), n_work, out, stream())
    return np.array(out[:6])


def _trace_vs_oracle(K, dK, NE, y, noise_e, noise_f, out):
    """out[2..4] of gprb_lml_eval (1/2 tr(W dK), 1/2 sum W_ii noise_i^2, 1/2 sum W_ii 2 noise_i) against the reference's
    algebra on the host (oracle.gp.lml_from_matrices), K + noise kept at cond <= 1e6.  Returns error / tolerance."""
    from oracle import gp as ogp
    Kh, dKh = K.cpu().numpy(), dK.cpu().numpy()
    noise = np.where(np.arange(len(Kh)) < NE, noise_e, noise_f)
    assert np.linalg.cond(Kh + np.diag(noise ** 2)) <= 1e6
    _, want = ogp.lml_from_matrices(Kh, np.dstack((dKh, np.diag(noise ** 2), np.diag(2 * noise))), y.cpu().numpy(), NE,
                                    noise_e, noise_f)
    ratio = np.abs(out[2:5] - want) / (1e-9 * np.abs(want) + 1e-9 * np.abs(want).max())
    assert ratio.max() <= 1.0, (out[2:5], want)
    return ratio.max()


def test_upper_mode_windows_symmetrize_and_trace(capsys):
    """The sharded build: every rank writes the J >= I blocks of its row window (FF_UPPER) into the full
    matrix, gprb_symmetrize mirrors them; the likelihood traces of gprb_lml_eval read dK right of the diagonal only."""
    from gpr_calculator_b200 import _lib, dist as gd
    from gpr_calculator_b200.device import Pack, k_total_device, build_force_rows, ptr, stream
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(11)
    X, dX, ELE, ind = list_to_tuple(make_force(rng, 37, lo=9, hi=41))
    f = Pack(X, ELE, ind, dxdr=dX)
    NF, N = 37, 3 * 37
    Kref, dKref = k_total_device(_lib.RBF, 1.1, 0.6, 2.0, (None, f), None, use_tol=False, grad=True, symmetric=False)
    y = torch.as_tensor(rng.normal(size=N), device="cuda")
    noise = 0.05
    full = _lml_eval(Kref, dKref, [(0, N)], 0, y, noise, noise)
    # (a) the entries left of the diagonal are never read: NaN there gives the same bits
    poisoned = torch.where(torch.triu(torch.ones(N, N, dtype=torch.bool, device="cuda")), dKref, float("nan"))
    assert np.array_equal(_lml_eval(Kref, poisoned, [(0, N)], 0, y, noise, noise), full)
    # (c) against the host
    margin = _trace_vs_oracle(Kref, dKref, 0, y, noise, noise, full)
    with capsys.disabled():
        print("\n[lml_eval traces, force rows] max |err| / tol vs host = %.2e" % margin)
    for parts in (1, 2, 3):
        windows = gd.row_windows([], ind, parts, upper=True)
        assert windows[0][1][0] == 0 and windows[-1][1][1] == NF
        K = torch.full((N, N), float("nan"), dtype=torch.float64, device="cuda")
        dK = torch.full((N, N), float("nan"), dtype=torch.float64, device="cuda")
        for (_, (f0, f1)) in windows:
            build_force_rows(_lib.RBF, 1.1, 0.6, 2.0, (None, f), (None, f), (f0, f1), K[3 * f0:3 * f1], dK[3 * f0:3 * f1],
                             use_tol=False, ff_mode=_lib.FF_UPPER)
        up = torch.triu(torch.ones(N, N, dtype=torch.bool, device="cuda"))
        assert (K - Kref)[up].abs().max().item() <= 1e-13 * Kref.abs().max().item()
        _lib.call("gprb_symmetrize", ptr(K), N, N, stream())
        assert (K - Kref).abs().max().item() <= 1e-13 * Kref.abs().max().item()
        # the FF_UPPER rows of dK (NaN left of the diagonal blocks) give the traces of the full dK
        got = _lml_eval(Kref, dK, [(0, N)], 0, y, noise, noise)
        assert np.all(np.abs(got[2:5] - full[2:5]) <= 1e-12 * np.abs(full[2:5]))


def test_trace_sharded_mode_and_transpose(capsys):
    """gprb_lml_eval reads K_ee (upper), K_fe and K_ff (upper) of dK only, and row ranges held by one rank give the traces of
    the whole matrix; gprb_transpose_copy fills K_ef from K_fe."""
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import Pack, k_total_device, stream, c_vp
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(21)
    X, dX, ELE, ind = list_to_tuple(make_force(rng, 17, lo=5, hi=30))
    Xe, Ee, inde = list_to_tuple(make_energy(rng, 6, lo=5, hi=30), mode="energy")
    f, e = Pack(X, ELE, ind, dxdr=dX), Pack(Xe, Ee, inde)
    K, dK = k_total_device(_lib.RBF, 1.2, 0.7, 2.0, (e, f), None, use_tol=False, grad=True)
    NE, N = 6, 6 + 51
    y = torch.as_tensor(rng.normal(size=N), device="cuda")
    noise_e, noise_f = 0.05, 0.1
    full = _lml_eval(K, dK, [(0, N)], NE, y, noise_e, noise_f)
    # (a) NaN in K_ef and left of the diagonal of K_ee and K_ff: never read, the same bits
    poisoned = dK.clone()
    poisoned[:NE, NE:] = float("nan")
    poisoned[NE:, NE:] = torch.where(torch.triu(torch.ones(N - NE, N - NE, dtype=torch.bool, device="cuda")), dK[NE:, NE:],
                                     torch.full_like(dK[NE:, NE:], float("nan")))
    poisoned[:NE, :NE] = torch.where(torch.triu(torch.ones(NE, NE, dtype=torch.bool, device="cuda")), dK[:NE, :NE],
                                     torch.full_like(dK[:NE, :NE], float("nan")))
    assert np.array_equal(_lml_eval(K, poisoned, [(0, N)], NE, y, noise_e, noise_f), full)
    # (b) four row ranges in one call, as a rank holds them (their rows stacked in dK_rows)
    ranges = [(0, 2), (2, NE), (NE, NE + 21), (NE + 21, N)]
    got = _lml_eval(K, poisoned, ranges, NE, y, noise_e, noise_f)
    assert np.all(np.abs(got[2:5] - full[2:5]) <= 1e-12 * np.abs(full[2:5]))
    # (c) against the host
    margin = _trace_vs_oracle(K, dK, NE, y, noise_e, noise_f, full)
    with capsys.disabled():
        print("\n[lml_eval traces, energy + force rows] max |err| / tol vs host = %.2e" % margin)
    Kt = K.clone()
    Kt[:NE, NE:] = float("nan")
    _lib.call("gprb_transpose_copy", c_vp(Kt.data_ptr() + NE * 8), N, c_vp(Kt.data_ptr() + NE * N * 8), N, N - NE, NE, stream())
    assert torch.equal(Kt, K) or (Kt - K).abs().max().item() <= 1e-15 * K.abs().max().item()


def test_flat_tiles_share_groups():
    """Groups that start and end in the middle of 8-row tiles and of 64-row CTA blocks on both sides,
    empty groups, and a row window that starts inside a tile."""
    from gpr_calculator_b200.kernels import rbf_kernel as rk
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import Pack, k_total_device
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(12)
    sizes1, sizes2 = [5, 1, 13, 64, 3, 97, 8, 7, 130, 2], [11, 96, 1, 1, 29, 63, 200, 5]
    mk = lambda sizes: list_to_tuple([make_force(rng, 1, lo=n, hi=n)[0] for n in sizes])   # noqa: E731
    F1, F2 = mk(sizes1), mk(sizes2)
    from oracle import kernels as ok
    O = ok.RBFOracle("port")
    for grad in (False, True):
        got, ref = rk.kff_C(F1, F2, 0.9, 0.8, 2.0, grad=grad), O.kff_C(F1, F2, 0.9, 0.8, 2.0, grad=grad)
        got, ref = (got, ref) if grad else ((got,), (ref,))
        for a, b in zip(got, ref):
            assert rel_err(a, b) <= TOL
    f1 = Pack(F1[0], F1[2], F1[3], dxdr=F1[1])
    f2 = Pack(F2[0], F2[2], F2[3], dxdr=F2[1])
    Kfull, _ = k_total_device(_lib.RBF, 0.9, 0.8, 2.0, (None, f1), (None, f2), use_tol=False)
    Kwin, _ = k_total_device(_lib.RBF, 0.9, 0.8, 2.0, (None, f1), (None, f2), use_tol=False, window=((0, 0), (2, 7)))
    assert torch.equal(Kwin, Kfull[6:21])
    # an empty group yields zero rows / columns
    Xe = np.concatenate((F1[0][:5], F1[0][5:]))
    g = Pack(Xe, F1[2], [5, 0, 1, 13, 64, 3, 97, 8, 7, 130, 2], dxdr=F1[1])
    Kg, _ = k_total_device(_lib.RBF, 0.9, 0.8, 2.0, (None, g), (None, f2), use_tol=False)
    assert torch.count_nonzero(Kg[3:6]).item() == 0 and torch.equal(Kg[6:], Kfull[3:]) and torch.equal(Kg[:3], Kfull[:3])


def test_kff_is_psd_and_deterministic():
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import Pack, k_total_device
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(8)
    X, dX, ELE, ind = list_to_tuple(make_force(rng, 60, lo=25, hi=34))
    f = Pack(X, ELE, ind, dxdr=dX)
    K1, _ = k_total_device(_lib.RBF, 1.0, 0.5, 2.0, (None, f), None, use_tol=True, tol=1e-10)
    K2, _ = k_total_device(_lib.RBF, 1.0, 0.5, 2.0, (None, f), None, use_tol=True, tol=1e-10)
    assert torch.equal(K1, K2)                              # fixed-order reductions: bitwise reproducible
    w = torch.linalg.eigvalsh(K1)
    assert w.min().item() >= -1e-9 * w.max().item()


def test_empty_groups_and_empty_sides(oracle_libs):
    """Groups without rows (a force centre with no neighbour inside rcut) give zero rows / columns, and
    a side without groups gives an empty block, like the reference's loops."""
    from gpr_calculator_b200.kernels import rbf_kernel as rk, dot_kernel as dk
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(11)
    d = 30

    def with_holes(items, holes):
        out = list(items)
        for h in holes:
            proto = out[0]
            empty = tuple(np.zeros((0,) + a.shape[1:], dtype=a.dtype) for a in proto)
            out.insert(h, empty)
        return out

    F1 = list_to_tuple(with_holes(make_force(rng, 5, lo=3, hi=20), (0, 3, 7)))
    F2 = list_to_tuple(with_holes(make_force(rng, 4, lo=3, hi=20), (2,)))
    # (an energy item is a whole structure: never empty -- the reference would divide by its zero atom count)
    E1 = list_to_tuple(make_energy(rng, 3, lo=3, hi=20), mode="energy")
    assert F1[-1].count(0) == 3 and F2[-1].count(0) == 1
    O, OD = oracle_libs.RBFOracle("port"), oracle_libs.DotOracle("port")
    for grad in (False, True):
        for fn_g, fn_o, a, b in ((rk.kff_C, O.kff_C, F1, F2), (rk.kef_C, O.kef_C, E1, F1), (rk.kee_C, O.kee_C, E1, E1)):
            got, ref = fn_g(a, b, 1.2, 0.8, 2.0, grad=grad), fn_o(a, b, 1.2, 0.8, 2.0, grad=grad)
            got, ref = (got, ref) if grad else ((got,), (ref,))
            for x, y in zip(got, ref):
                assert x.shape == y.shape and np.all(np.isfinite(x)) and rel_err(x, y) <= TOL
    K = rk.kff_C(F1, F2, 1.2, 0.8, 2.0)
    assert np.all(K[0:3] == 0) and np.all(K[9:12] == 0) and np.all(K[21:24] == 0) and np.all(K[:, 6:9] == 0)
    assert rel_err(dk.kff_C(F1, F2, 2.0, 1.5, 3.0), OD.kff_C(F1, F2, 2.0, 1.5, 3.0)) <= TOL
    # a side with no groups at all
    none = (np.zeros((0, d)), np.zeros((0, d, 3)), np.zeros(0, dtype=int), [])
    assert rk.kff_C(none, F2, 1.2, 0.8, 2.0).shape == (0, 3 * len(F2[-1]))
    assert rk.kff_C(F2, none, 1.2, 0.8, 2.0).shape == (3 * len(F2[-1]), 0)


def test_properties_at_profiling_size():
    """Size-independent properties on a real descriptor workload (100 x Cu32 from the device SO3, N = 9 700):
    K = K^T, K(sigma) = sigma^2 K(1), dK/dl = central difference of K in l, diag mode = diagonal, and the
    row-window build reproduces the one-pass build."""
    from gpr_calculator_b200 import _lib, synthetic as syn
    from gpr_calculator_b200.device import Pack, k_total_device, diag_device
    from gpr_calculator_b200.SO3 import SO3
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in syn.structures(100, 2, 2000)])
    e = Pack(E_dev[0], E_dev[1], E_dev[2])
    f = Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])
    NE, NF = e.n_groups, f.n_groups
    sig, ell = 1.0, 0.1
    K, dK = k_total_device(_lib.RBF, sig, ell, 2.0, (e, f), None, use_tol=False, grad=True)
    N = NE + 3 * NF
    assert K.shape == (N, N) and bool(torch.isfinite(K).all()) and bool(torch.isfinite(dK).all())
    scale = K.abs().max().item()
    assert (K - K.T).abs().max().item() <= 1e-13 * scale and (dK - dK.T).abs().max().item() <= 1e-13 * dK.abs().max().item()
    K2, _ = k_total_device(_lib.RBF, 3.0 * sig, ell, 2.0, (e, f), None, use_tol=False, grad=False)
    assert (K2 - 9.0 * K).abs().max().item() <= 1e-13 * 9.0 * scale
    h = 1e-6
    Kp, _ = k_total_device(_lib.RBF, sig, ell + h, 2.0, (e, f), None, use_tol=False, grad=False)
    Km, _ = k_total_device(_lib.RBF, sig, ell - h, 2.0, (e, f), None, use_tol=False, grad=False)
    fd = (Kp - Km) / (2 * h)
    assert (fd - dK).abs().max().item() <= 1e-6 * dK.abs().max().item()
    dg = diag_device(_lib.RBF, sig, ell, 2.0, (None, f), tol=0.0)
    assert (dg - torch.diagonal(K)[NE:]).abs().max().item() <= 1e-13 * scale
    w = ((10, 30), (700, 1500))
    Kw, _ = k_total_device(_lib.RBF, sig, ell, 2.0, (e, f), None, use_tol=False, grad=False, window=w)
    ref = torch.cat((K[10:30], K[NE + 3 * 700:NE + 3 * 1500]))
    assert (Kw - ref).abs().max().item() <= 1e-13 * scale


def test_two_stage_path_matches_block_path(monkeypatch):
    """The two-stage contraction (default for the no-gradient K_ff at d = 29..32) against the 4x4-block kernel
    (GPRB_KFF_TWO_STAGE=0): ragged groups, three species, pair cut, full / symmetric / upper modes, RBF and Dot."""
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import Pack, k_total_device
    from gpr_calculator_b200.utilities import list_to_tuple
    rng = np.random.default_rng(21)
    X, dX, ELE, ind = list_to_tuple(make_force(rng, 37, lo=3, hi=40, species=(1, 16, 46), zero_rows=1))
    f = Pack(X, ELE, ind, dxdr=dX)
    X2, dX2, ELE2, ind2 = list_to_tuple(make_force(rng, 23, lo=1, hi=70, species=(1, 16, 46)))
    f2 = Pack(X2, ELE2, ind2, dxdr=dX2)
    for kern, p1, zeta in ((_lib.RBF, 0.7, 2.0), (_lib.RBF, 0.4, 3.0), (_lib.DOT, 1.1, 2.0)):
        for side2, sym, tol in ((None, True, 1e-10), (None, False, 1e-10), ((None, f2), False, 1e-3)):
            out = {}
            for two in ("", "1"):
                if two:
                    monkeypatch.delenv("GPRB_KFF_TWO_STAGE", raising=False)
                else:
                    monkeypatch.setenv("GPRB_KFF_TWO_STAGE", "0")
                out[two], _ = k_total_device(kern, 1.3, p1, zeta, (None, f), side2, use_tol=True, tol=tol, grad=False, symmetric=sym)
            scale = out[""].abs().max().item()
            assert (out["1"] - out[""]).abs().max().item() <= 1e-12 * scale


def test_kee_tensor_path_species_blocks(oracle_libs):
    """K_ee on the DMMA tile path in the shape of the Pd4/MgO training set: large energy groups whose rows are ordered by
    species (tiles without a same-species pair are skipped, also when a group ends inside a skipped tile), ragged group
    sizes, the symmetric training block and a rectangular window; against the C oracle."""
    from gpr_calculator_b200.kernels import rbf_kernel as rk, dot_kernel as dk
    rng = np.random.default_rng(77)
    base = np.abs(rng.normal(size=30)) + 0.5

    def side(sizes):
        X, ELE = [], []
        for n_mg, n_o, n_pd in sizes:
            n = n_mg + n_o + n_pd
            X.append(base[None, :] + 0.3 * rng.normal(size=(n, 30)))
            ELE.append(np.array([12] * n_mg + [8] * n_o + [46] * n_pd))
        return np.concatenate(X), np.concatenate(ELE), [sum(t) for t in sizes]
    E1 = side([(108, 108, 4), (108, 108, 4), (50, 61, 1), (3, 0, 9), (0, 17, 0), (108, 108, 4)])
    E2 = side([(20, 30, 4), (108, 108, 4), (1, 1, 1)])
    O, OD = oracle_libs.RBFOracle("port"), oracle_libs.DotOracle("port")
    for a, b in ((E1, E1), (E1, E2), (E2, E1)):
        for zeta in (2.0, 3.0):
            ref = O.kee_C(a, b, 1.4, 0.35, zeta, grad=True)
            got = rk.kee_C(a, b, 1.4, 0.35, zeta, grad=True)
            for x, y in zip(got, ref):
                assert x.shape == y.shape and rel_err(x, y) <= TOL, zeta
            assert rel_err(dk.kee_C(a, b, 2.0, 1.5, zeta), OD.kee_C(a, b, 2.0, 1.5, zeta)) <= TOL
    K = rk.kee_C(E1, E1, 1.4, 0.35, 2.0)
    assert np.array_equal(K, K.T)
