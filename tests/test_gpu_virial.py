"""GPU: total stress of batches of structures from one row per atom (gprb_virial_rows, device.k_virial_device,
GP.predict_structures(stress=True), GPR(stress_std=True)).

- The kernel against a numpy segmented sum of rdxdr in the same order, on Cu32 and Pd4/MgO structures; two calls bitwise.
- The merge is exact: every virial K* row equals the sum over the structure's atoms of the per-atom stress rows of
  k_total_stress_device, and the virial prior equals the sum of the per-atom stress packs' FF_FULL self-block (RBF at
  zeta = 2 and 3, Dot).  Each entry is held to 1e-12 of the Cauchy-Schwarz scale of the per-atom terms it sums,
  sum_a sqrt(k_aa k_jj): shear components of near-cubic environments cancel between atoms, so the summed value itself
  can be far below the magnitude the per-atom route rounds at.
- Means against predict_structure(stress=True)[2].sum(0); E, F and their sigma bitwise those of stress=False.
- sigma against a host reference k(S,S) - k*^T (K + noise)^-1 k* with N = 2 328 real Cu32 rows.
- Sharded against shard=False on >= 2 GPUs, and the calculator's stress_std option."""
import io
import os
import contextlib
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOIGT = [0, 4, 8, 1, 2, 5]


def _des():
    from gpr_calculator_b200.SO3 import SO3
    return SO3(nmax=3, lmax=4, rcut=5.0, stress=True)


def _cu(n, seed0, fixed=None):
    from gpr_calculator_b200 import synthetic as syn
    from gpr_calculator_b200.utilities import FixAtoms
    out = [a for a, _, _ in syn.structures(n, 2, seed0)]
    if fixed is not None:
        out[0].constraints = [FixAtoms(fixed)]
    return out


def _pd4(ids):
    from gpr_calculator_b200.utilities import SimpleAtoms
    g = np.load(os.path.join(GOLD, "pd4.npz"))
    return [SimpleAtoms(g["numbers"], g["positions"][k], g["cell"], g["pbc"]) for k in ids]


def _segmented_sum(r):
    """numpy: per atom, the Voigt columns of rdxdr summed over its seq rows in increasing q."""
    rd = r["rdxdr"].cpu().numpy()
    rd = rd.reshape(rd.shape[0], rd.shape[1], 9)[:, :, VOIGT]
    sp = r["seq_ptr"].cpu().numpy().astype(np.int64)
    cnt = sp[1:] - sp[:-1]
    out = np.zeros((len(cnt), rd.shape[1], 6))
    for j in range(int(cnt.max())):
        a = np.nonzero(cnt > j)[0]
        out[a] = out[a] + rd[sp[a] + j]
    return out


def test_virial_rows_kernel_vs_numpy():
    from gpr_calculator_b200.batch import virial_rows_from_batch
    des = _des()
    for atoms in (_cu(3, 3000), _pd4([0, 100])):
        r = des.calculate_batch(atoms, to_host=False)
        E, (X, V, ele, ind) = virial_rows_from_batch(r)
        assert ind == [len(a) for a in atoms] and E[2] == ind and torch.equal(X, r["x"]) and X.shape[0] == V.shape[0]
        assert torch.equal(ele, r["numbers"].to(torch.int32))
        ref = _segmented_sum(r)
        assert rel_err(V.cpu().numpy(), ref) <= 1e-15
        assert torch.equal(virial_rows_from_batch(r)[1][1], V)


def _train_packs(des, atoms):
    from gpr_calculator_b200 import device as gdev, synthetic as syn
    E, F = syn.packed_from_batch(des, atoms)
    return gdev.Pack(E[0], E[1], E[2]), gdev.Pack(F[0], F[2], F[3], dxdr=F[1])


def _per_atom_reference(kernel, r, train, f_tol, prior_norm_eps, prior_zeta, prior_tol):
    """Per-atom stress route summed over the atoms of each structure: K* [6 S, N], prior [6 S], and the per-atom
    Cauchy-Schwarz scales of both sums (sum_a sqrt(k_aa) per structure and Voigt component)."""
    from gpr_calculator_b200 import _lib, device as gdev
    from gpr_calculator_b200.batch import rows_from_batch
    E_t, F_t = rows_from_batch(r, None, stress=True)
    f1, sa, sb = gdev.stress_packs(F_t)
    _, K1 = kernel.k_total_stress_device({"energy": gdev.energy_pack(E_t), "force": (f1, sa, sb)}, train, tol=f_tol)
    counts = E_t[2]
    S, A = len(counts), sum(counts)
    grp = np.repeat(np.arange(S), counts)
    K1 = K1.cpu().numpy().reshape(A, 6, -1)
    Ks = np.zeros((S, 6, K1.shape[2]))
    np.add.at(Ks, grp, K1)
    prior, scale = np.zeros((S, 6)), np.zeros((S, 6))
    p0, p1 = (kernel.sigma, kernel.l) if kernel.name == "RBF" else (kernel.sigma, kernel.sigma0)
    kid = _lib.RBF if kernel.name == "RBF" else _lib.DOT
    for t, a in enumerate((0, 3)):
        P = gdev.Pack(F_t[0], F_t[2], F_t[3], dxdr=F_t[1][:, :, 3 + a:6 + a], norm_eps=prior_norm_eps)
        Kf = torch.empty((3 * A, 3 * A), dtype=torch.float64, device="cuda")
        _lib.call("gprb_kff", kid, P.handle, P.handle, float(p0), float(p1), float(prior_zeta), 1, float(prior_tol),
                  _lib.FF_FULL, 0, A, gdev.ptr(Kf), 3 * A, gdev.c_vp(0), 0, gdev.stream())
        Kf = Kf.cpu().numpy().reshape(A, 3, A, 3)
        d = np.sqrt(np.abs(np.einsum("acac->ac", Kf)))
        for s in range(S):
            m = grp == s
            prior[s, 3 * t:3 * t + 3] = np.einsum("acbc->c", Kf[m][:, :, m])
            scale[s, 3 * t:3 * t + 3] = d[m].sum(0)
    return Ks.reshape(6 * S, -1), prior.reshape(-1), scale.reshape(-1)


@pytest.mark.parametrize("case", ["rbf_zeta2", "rbf_zeta3", "dot"])
def test_virial_kstar_and_prior_equal_summed_per_atom_rows(case):
    from gpr_calculator_b200.batch import virial_rows_from_batch
    from gpr_calculator_b200.kernels import RBF_mb, Dot_mb
    des = _des()
    if case == "dot":
        kernel, f_tol, eps, zp, tp = Dot_mb(para=[2.0, 1.5], zeta=3), 0.0, 1e-8, 3.0, 0.0
    else:
        zeta = 2.0 if case == "rbf_zeta2" else 3.0
        kernel, f_tol, eps, zp, tp = RBF_mb(para=[1.0, 0.5], zeta=zeta), 1e-10, 0.0, zeta, 1e-12
    for train_atoms, test_atoms in ((_cu(6, 2000), _cu(3, 3000)), (_pd4([0, 50, 150]), _pd4([10, 200]))):
        e2, f2 = _train_packs(des, train_atoms)
        train = {"energy": e2, "force": f2}
        d_train = kernel.diag_device(train, _packed_ok=True).cpu().numpy()
        r = des.calculate_batch(test_atoms, to_host=False)
        Ks, prior = kernel.k_virial_device(virial_rows_from_batch(r)[1], train, tol=f_tol)
        Ks, prior = Ks.cpu().numpy(), prior.cpu().numpy()
        Ks_ref, prior_ref, s_row = _per_atom_reference(kernel, r, train, f_tol, eps, zp, tp)
        assert Ks.shape == Ks_ref.shape == (6 * len(test_atoms), len(d_train))
        err_k = float((np.abs(Ks - Ks_ref) / (np.outer(s_row, np.sqrt(np.abs(d_train))) + 1e-300)).max())
        err_p = float((np.abs(prior - prior_ref) / (s_row ** 2 + 1e-300)).max())
        strict = float((np.abs(prior - prior_ref) / (np.abs(prior_ref) + 1e-300)).max())
        print("[virial %s] K* %.2e prior %.2e (relative to the summed prior %.2e)" % (case, err_k, err_p, strict))
        assert err_k <= 1e-12 and err_p <= 1e-12
        assert np.all(prior > 0)


def _fitted_gp(n_train=24, kernel=None):
    from gpr_calculator_b200 import synthetic as syn
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    des = _des()
    labelled = syn.structures(n_train, 2, 2000)
    e_pack, f_pack = _train_packs(des, [a for a, _, _ in labelled])
    gp = GP(kernel=kernel or RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    gp.train_x = {"energy": e_pack, "force": f_pack}
    y = syn.targets(labelled)
    gp.train_y = {"energy": list(y[:n_train, 0]), "force": y[n_train:, 0].reshape(-1, 3)}
    gp.N_energy, gp.N_forces = n_train, n_train * 32
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(opt=False, show=False)
    return gp


def test_predict_structures_stress_means():
    gp = _fitted_gp(8)
    tests_ = _cu(5, 3000, fixed=[0, 3, 7])
    plain = gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=3)
    got = gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=3, stress=True)
    mean_only = gp.predict_structures(tests_, f_tol=1e-12, batch=3, stress=True)
    assert len(got) == len(tests_)
    for st_, a, b, m in zip(tests_, got, plain, mean_only):
        assert len(a) == 6 and a[2].shape == (6,) and a[5].shape == (6,) and np.all(np.isfinite(a[5]))
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and a[3] == b[3] and np.array_equal(a[4], b[4])
        assert len(m) == 3 and m[0] == a[0] and np.array_equal(m[2], a[2])
        S_ref = gp.predict_structure(st_, stress=True, f_tol=1e-12)[2].sum(axis=0)
        assert rel_err(a[2], S_ref) <= 1e-10
    from gpr_calculator_b200.SO3 import SO3
    gp.descriptor = SO3(nmax=3, lmax=4, rcut=5.0)                # no rdxdr: loud, as predict_structure(stress=True)
    with pytest.raises(ValueError):
        gp.predict_structures(tests_[:1], stress=True)


@pytest.mark.timeout(900)
def test_stress_sigma_against_reference(monkeypatch, capsys):
    from scipy.linalg import cho_factor, cho_solve
    from gpr_calculator_b200.batch import virial_rows_from_batch
    from test_gpu_gp import _sigma_reference_formula, _sigma_refined
    gp = _fitted_gp(24)                                    # N = 24 + 2 304 = 2 328
    tests_ = _cu(20, 3000)
    r = gp.descriptor.calculate_batch(tests_, to_host=False)
    Ks, prior, _ = _per_atom_reference(gp.kernel, r, gp.train_x, 1e-12, 0.0, 2.0, 1e-12)
    Kn, _ = gp.kernel.k_total_device(gp.train_x, None, f_tol=1e-10, grad=False)
    Kn = Kn.cpu().numpy()
    idx = np.arange(len(Kn))
    Kn[idx, idx] += np.where(idx < 24, 0.002 ** 2, 0.1 ** 2)
    c = cho_factor(Kn, lower=True)
    var = prior - np.einsum("ij,ji->i", Ks, cho_solve(c, Ks.T))
    sig_cho = np.sqrt(np.maximum(var, 0.0))
    sig_ref, L = _sigma_reference_formula(Kn, Ks, prior)
    sig_true = _sigma_refined(L, Kn, Ks, prior)
    got = {}
    for route in ("chol", "inverse"):
        monkeypatch.setenv("GPRB_VARIANCE_ROUTE", route)
        res = gp.predict_structures(tests_, return_std=True, f_tol=1e-12, batch=10, stress=True)
        got[route] = np.concatenate([t[5] for t in res])
    monkeypatch.delenv("GPRB_VARIANCE_ROUTE")
    assert virial_rows_from_batch(r)[1][1].shape[0] == 32 * 20
    err_chol = float((np.abs(got["chol"] - sig_cho) / np.sqrt(prior)).max())
    floor = max(1e-8, 4.0 * np.abs(sig_ref - sig_true).max())
    err_inv = float(np.abs(got["inverse"] - sig_ref).max())
    with capsys.disabled():
        print("\n[stress sigma] N = %d, m = %d, sigma %.3g .. %.3g; chol route vs cho_solve %.3e of sqrt k(S,S); "
              "inverse route vs reference formula %.3e (floor %.3e)"
              % (len(Kn), len(prior), sig_cho.min(), sig_cho.max(), err_chol, err_inv, floor))
    assert err_chol <= 1e-9
    assert err_inv <= floor


def test_gpr_calculator_stress_std():
    from gpr_calculator_b200.calculator import GPR
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.synthetic import cu_fcc
    gp = GP(kernel=RBF_mb(para=[1.0, 0.5], zeta=2.0), descriptor=SO3(nmax=3, lmax=4, rcut=4.0, stress=True),
            noise_e=0.002, noise_f=0.05, log_file=None)
    for k in (1, 2):
        at, E, F = cu_fcc(1, k, noise=0.08)
        gp.add_structure((at, E, F))
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(show=False)
    at = cu_fcc(1, 7, noise=0.08)[0]
    res = {}
    for opt in (False, True):
        calc = GPR(base=None, ff=gp, save=False, stress=True, **({"stress_std": True} if opt else {}))
        calc.freeze()
        calc.update_gpr = False
        with contextlib.redirect_stdout(io.StringIO()):
            calc.calculate(at.copy())
        res[opt] = dict(calc.results)
        if opt:
            assert np.array_equal(calc.get_var_s(), calc.results["var_s"])
    E, F, S, E_std, F_std = gp.predict_structure(at.copy(), stress=True, return_std=True, f_tol=1e-12)
    old = res[False]
    assert "var_s" not in old and old["energy"] == E and np.array_equal(old["forces"], F)
    assert np.array_equal(old["stress"], S.sum(axis=0)) and old["var_e"] == E_std and np.array_equal(old["var_f"], F_std)
    new = res[True]
    assert new["stress"].shape == (6,) and new["var_s"].shape == (6,) and np.all(np.isfinite(new["var_s"]))
    assert np.all(new["var_s"] >= 0) and rel_err(new["stress"], old["stress"]) <= 1e-10
    assert abs(new["energy"] - old["energy"]) <= 1e-9 and np.abs(new["forces"] - old["forces"]).max() <= 1e-9
    assert "var_s" in GPR.implemented_properties


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(600)
def test_sharded_stress_predictions_match_unsharded():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    n = min(n, 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "multi_gpu_virial_worker.py")]
    res = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=580)
    assert res.returncode == 0, res.stdout[-6000:]
