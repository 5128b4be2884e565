"""GPU parity of the GP API (set_train_pts / fit / log_marginal_likelihood / predict_structure)
against golden vectors produced by the reference GP.  Tolerances (north_star): predicted E and F
within 1e-8 eV (eV/A); sigma within the conditioning bound explained in test_oracle_golden.py."""
import io
import os
import contextlib

import numpy as np
import pytest
from scipy.optimize import approx_fprime

from helpers import rel_err
from test_oracle_golden import std_tolerance

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLD, "gp.npz"))


def _atoms(g, pos, fixed=True):
    from gpr_calculator_b200.utilities import SimpleAtoms, FixAtoms
    return SimpleAtoms(g["numbers"], pos, g["cell"], g["pbc"], constraints=[FixAtoms(g["fixed"])] if fixed else [])


def _model(g, kernel="RBF"):
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb, Dot_mb
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.utilities import convert_train_data
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    labelled = [(_atoms(g, g["t%d_pos" % k]), float(g["t%d_E" % k]), g["t%d_F" % k]) for k in range(3)]
    tdata = convert_train_data(labelled, des)
    ker = RBF_mb(para=[1.0, 0.1], zeta=2.0) if kernel == "RBF" else Dot_mb(para=[2, 2.0], zeta=2.0)
    gp = GP(kernel=ker, descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(TrainData=tdata, opt=False, show=False)
    return gp


def test_lml_and_gradient_vs_golden(g):
    gp = _model(g)
    assert len(gp.y_train) == int(g["N"]) and np.allclose(gp.y_train, g["y_train"], atol=1e-13, rtol=0)
    for tag, prm in (("a", [1.0, 0.1]), ("b", [2.0, 0.8])):
        lml, grad = gp.log_marginal_likelihood(np.array(prm), eval_gradient=True)
        assert abs(lml - g["lml_" + tag]) <= 1e-8 * abs(g["lml_" + tag])
        assert rel_err(grad, g["lml_grad_" + tag]) <= 1e-6
        assert abs(gp.log_marginal_likelihood(np.array(prm)) - lml) <= 1e-6 * abs(lml)   # tol-cut K vs uncut
    # the analytic gradient is a true derivative
    f = lambda p: gp.log_marginal_likelihood(np.array(p))   # noqa: E731
    _, grad = gp.log_marginal_likelihood(np.array([2.0, 0.8]), eval_gradient=True)
    fd = approx_fprime(np.array([2.0, 0.8]), f, 1e-6)
    assert rel_err(grad, fd) <= 1e-4


def test_fit_and_predict_structure_vs_golden(g):
    gp = _model(g)
    gp.kernel.update([2.0, 0.8])
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(opt=False, show=False)
    assert rel_err(gp.kernel.k_total(gp.train_x), g["K_b"]) <= 1e-10
    assert rel_err(gp.alpha_, g["alpha_b"]) <= 1e-6
    L = gp.L_
    K = g["K_b"].copy()
    K[np.arange(3), np.arange(3)] += 0.002 ** 2
    K[np.arange(3, len(K)), np.arange(3, len(K))] += 0.1 ** 2
    assert rel_err(L @ L.T, K) <= 1e-12
    assert rel_err(gp._K_inv @ K, np.eye(len(K))) <= 1e-6
    test = _atoms(g, g["test_pos"])
    E, F, S, E_std, F_std = gp.predict_structure(test, stress=False, return_std=True, f_tol=1e-12)
    assert S is None
    assert abs(E - g["pred_E"]) <= 1e-8 and np.abs(F - g["pred_F"]).max() <= 1e-8
    assert np.all(F[g["fixed"]] == 0) and np.all(F_std[g["fixed"]] == 0)      # FixAtoms rows are dropped
    bound = std_tolerance(g["K_b"], 0.002, 0.1, 3, np.array([4.0]))
    assert abs(E_std ** 2 - g["pred_E_std"] ** 2) <= bound
    assert np.abs(F_std ** 2 - g["pred_F_std"] ** 2).max() <= bound
    Ev, Ep, Fv, Fp = gp.validate_data()
    assert np.abs(Ep - g["val_E_pred"]).max() <= 1e-8 and np.abs(Fp - g["val_F_pred"]).max() <= 1e-8
    # packed-tuple diag works here (the reference truncates it, RBF_mb.py:87) and stds are finite
    out = gp.validate_data(return_std=True)
    assert np.all(np.isfinite(out[2])) and np.all(np.isfinite(out[5]))
    E2, F2, _ = gp.predict_structure(test, stress=False)
    assert E2 == E and np.array_equal(F2, F)
    with pytest.raises(ValueError):
        gp.predict_structure(test)            # reference default stress=True needs SO3(stress=True) (tests/test_stress.py)


def test_optimisation_trajectory_vs_golden(g):
    """L-BFGS-B from the reference's initial guess: same printed Loss lines (3 decimals) and the same
    optimum."""
    gp = _model(g)
    gp.kernel.update([1.0, 0.1])
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        gp.fit(opt=True, show=True, maxiter=10)
    lines = [ln for ln in buf.getvalue().splitlines() if ln.startswith("Loss:")]
    trace = np.array([[float(v) for v in ln.split()[1:]] for ln in lines])
    assert trace.shape == g["opt_trace"].shape
    assert np.abs(trace - g["opt_trace"]).max() <= 2e-3          # printed with 3 decimals
    assert rel_err(np.array(gp.kernel.parameters()), g["opt_params"]) <= 1e-5
    test = _atoms(g, g["test_pos"])
    E, F, S, E_std, F_std = gp.predict_structure(test, stress=False, return_std=True, f_tol=1e-12)
    assert abs(E - g["opt_pred_E"]) <= 1e-6 and np.abs(F - g["opt_pred_F"]).max() <= 1e-6
    assert gp.fits == 2 and gp.N_queue == 0


def test_dot_gp_vs_golden(g):
    gp = _model(g, kernel="Dot")
    lml, grad = gp.log_marginal_likelihood(np.array([2.0, 2.0]), eval_gradient=True)
    assert abs(lml - g["dot_lml"]) <= 1e-8 * abs(g["dot_lml"])
    assert rel_err(grad, g["dot_lml_grad"]) <= 1e-6
    assert rel_err(gp.alpha_, g["dot_alpha"]) <= 1e-6


def test_add_structure_selection_and_refit(g):
    """add_structure on an untrained and a trained model: energy always added, force centres
    capped at N_max and de-duplicated; queue counters; refit clears the queue."""
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    gp = GP(kernel=RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=SO3(nmax=3, lmax=4, rcut=5.0),
            noise_e=0.002, noise_f=0.1, log_file=None)
    at0 = _atoms(g, g["t0_pos"], fixed=False)
    pts, n, err = gp.add_structure((at0, float(g["t0_E"]), g["t0_F"].copy()))
    assert n == 1 + len(pts["force"]) and 1 <= len(pts["force"]) <= 13
    assert gp.N_energy == 1 and gp.N_queue == n
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(show=False)
    assert gp.N_queue == 0 and gp.alpha_ is not None
    at1 = _atoms(g, g["t1_pos"], fixed=False)
    pts, n, err = gp.add_structure((at1, float(g["t1_E"]), g["t1_F"].copy()), N_max=3)
    assert len(pts["force"]) <= 3 and gp.N_energy == 2 and gp.N_queue == n
    # predictions use only the fitted part of the training set while points wait in the queue
    E, F, _ = gp.predict_structure(at1, stress=False)
    assert np.isfinite(E) and np.all(np.isfinite(F))


def test_gpr_calculator_adapter(capsys):
    """GPR(base=..., ff=...) control flow (calculator.py:48-117): uncertain structures go to the base
    calculator and enter the training queue, confident ones use the surrogate, the model is refitted
    on the reference's cadence; result keys and printed lines as in the reference."""
    from gpr_calculator_b200.calculator import GPR
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.synthetic import cu_fcc, K_SPRING, A_CU

    class Einstein:
        """toy base calculator: harmonic wells on the fcc sites"""
        def __init__(self):
            self.site = cu_fcc(1, 0, noise=0.0)[0].positions
        def get_potential_energy(self, atoms):
            return 0.5 * K_SPRING * float(((atoms.positions - self.site) ** 2).sum())
        def get_forces(self, atoms):
            return -K_SPRING * (atoms.positions - self.site)

    base = Einstein()
    gp = GP(kernel=RBF_mb(para=[1.0, 0.5], zeta=2.0), descriptor=SO3(nmax=3, lmax=4, rcut=4.0),
            noise_e=0.002, noise_f=0.05, log_file=None)
    first = cu_fcc(1, 1, noise=0.08)[0]
    first.calc = base
    gp.add_structure((first.copy(), base.get_potential_energy(first), base.get_forces(first)))
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(show=False)
    calc = GPR(base=base, ff=gp, save=False, freq=2)
    for k in range(2, 7):
        at = cu_fcc(1, k, noise=0.08)[0]
        calc.calculate(at)
        assert set(("energy", "forces", "var_e", "var_f")) <= set(calc.results)
        assert calc.results["forces"].shape == (4, 3) and np.isfinite(calc.results["energy"])
    out = capsys.readouterr().out
    assert "From Base model" in out or "From Surrogate" in out
    assert gp.use_base + gp.use_surrogate == 5
    calc.force_base = True                   # two labelled structures in the queue trigger a refit (calculator.py:102)
    n_fits = gp.fits
    for k in (50, 51):
        calc.calculate(cu_fcc(1, k, noise=0.08)[0])
    calc.force_base = False
    assert gp.use_base >= 2 and gp.fits >= n_fits + 1 and gp.N_energy_queue < 2
    assert calc.get_e(peratom=False) == calc.results["energy"] and calc.get_var_f().shape == (4, 3)
    calc.freeze()
    n_base = gp.use_base
    calc.calculate(cu_fcc(1, 99, noise=0.3)[0])
    assert gp.use_base == n_base             # frozen: the base calculator is not called


def _oracle_lml(gp, theta):
    """oracle.gp.lml_from_matrices on the noise-free K (and dK/dl) the GP builds on device, with the gradient components of
    GP.log_marginal_likelihood: 2K/sigma, then dK/dl (RBF) or the E-E constant d/dsigma0 of dot_kernel.py:58 (Dot), then
    diag(2 noise_i) when the noise is a hyper-parameter (gaussianprocess.py:196-198)."""
    from oracle import gp as ogp
    ker = gp.kernel
    ker.update(theta if gp.noise_bounds is None else theta[:-1])
    Kd, dKd = ker.k_total_device(gp.train_x, None, f_tol=1e-10, grad=True)
    K = Kd.cpu().numpy()
    NE = gp._n_energy_rows()
    if dKd is not None:
        dK = dKd.cpu().numpy()
    else:
        dK = np.zeros_like(K)
        dK[:NE, :NE] = 0.8 * 2 * ker.sigma ** 2 * ker.sigma0
    comps = [2 * K / ker.sigma, dK]
    noise_e, noise_f = gp.noise_e, gp.noise_f
    if gp.noise_bounds is not None:
        noise_e, noise_f = theta[-1], gp.f_coef * theta[-1]
        comps.append(np.diag(np.where(np.arange(len(K)) < NE, 2 * noise_e, 2 * noise_f)))
    return ogp.lml_from_matrices(K, np.dstack(comps), gp.y_train, NE, noise_e, noise_f)


def test_inverse_rows_and_gradient_routes(g):
    """gprb_chol_inverse_rows against numpy (trailing-block solves), and the likelihood and its gradient (blocked
    inverse-rows route of gprb_lml_eval) against the reference's algebra evaluated on the host on the same K and dK
    (explicit inverse, gaussianprocess.py:195)."""
    import torch
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import ptr, stream
    rng = np.random.default_rng(4)
    N = 257
    A = rng.normal(size=(N, N))
    K = A @ A.T + N * np.eye(N)
    ref = np.linalg.inv(K)
    Kd = torch.as_tensor(K, device="cuda").contiguous()
    _lib.call("gprb_chol_factor", ptr(Kd), N, N, stream())
    for (r0, r1, c0) in ((0, 17, 0), (40, 97, 40), (40, 97, 11), (200, 257, 200), (256, 257, 256), (5, 5, 5)):
        out = torch.full((max(r1 - r0, 1), N - c0 + 3), 7.0, dtype=torch.float64, device="cuda")     # padded leading dimension
        _lib.call("gprb_chol_inverse_rows", ptr(Kd), N, N, r0, r1, c0, ptr(out), N - c0 + 3, stream())
        if r1 > r0:
            assert rel_err(out[:, :N - c0].cpu().numpy(), ref[r0:r1, c0:]) <= 1e-10
            assert bool((out[:, N - c0:] == 7.0).all())
    cases = [("RBF", np.array([1.3, 0.25]), None), ("Dot", np.array([2.0, 1.5]), None),
             # a noise hyper-parameter adds the third gradient component (noise_bounds, gaussianprocess.py:196-198)
             ("RBF", np.array([1.3, 0.25, 0.004]), [1e-4, 1e-1])]
    for kernel, theta, noise_bounds in cases:
        gp = _model(g, kernel)
        gp.noise_bounds = noise_bounds
        lml, grad = gp.log_marginal_likelihood(theta, eval_gradient=True)
        lml_h, grad_h = _oracle_lml(gp, theta)
        assert len(grad) == len(theta)
        assert abs(lml - lml_h) <= 1e-12 * abs(lml_h), (kernel, lml, lml_h)
        assert np.allclose(grad, grad_h, rtol=1e-9, atol=1e-9 * np.abs(grad_h).max()), (kernel, grad, grad_h)


def _inverse_as_set_K_inv(Ld, N):
    """K^-1 from the factor the way GP.set_K_inv forms it: rows right of the diagonal by trailing-block solves, then mirrored."""
    import torch
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import c_vp, ptr, stream
    Kinv = torch.empty((N, N), dtype=torch.float64, device="cuda")
    for r0, r1 in ((0, N // 3), (N // 3, N)):
        _lib.call("gprb_chol_inverse_rows", ptr(Ld), N, N, r0, r1, r0, c_vp(Kinv.data_ptr() + (r0 * N + r0) * 8), N, stream())
    _lib.call("gprb_symmetrize", ptr(Kinv), N, N, stream())
    return Kinv


def test_variance_routes_match_numpy(g, monkeypatch):
    """Predictive variance through the explicit inverse (gprb_predict, the reference's formula) and through the Cholesky
    factor (gprb_predict_chol, used for batches) against numpy, and the two routes through GP.predict_structures."""
    import torch
    from gpr_calculator_b200 import _lib
    from gpr_calculator_b200.device import ptr, stream
    rng = np.random.default_rng(8)
    N, m = 300, 41
    A = rng.normal(size=(N, N))
    K = A @ A.T + N * np.eye(N)
    Ks = rng.normal(size=(m, N + 5))[:, :N]                 # rows with a leading dimension > N
    alpha = rng.normal(size=N)
    prior = 10.0 + rng.uniform(size=m)
    quad = np.einsum("ij,ij->i", Ks @ np.linalg.inv(K), Ks)
    want_var = np.maximum(prior - quad, 0.0)
    Ld = torch.as_tensor(K, device="cuda").contiguous()
    _lib.call("gprb_chol_factor", ptr(Ld), N, N, stream())
    Kinv = _inverse_as_set_K_inv(Ld, N)
    Kd = torch.as_tensor(np.ascontiguousarray(rng.normal(size=(m, N + 5))), device="cuda")
    Kd[:, :N] = torch.as_tensor(Ks, device="cuda")
    ad, dd = torch.as_tensor(alpha, device="cuda"), torch.as_tensor(prior, device="cuda")
    for name in ("gprb_predict", "gprb_predict_chol"):
        mean = torch.empty(m, dtype=torch.float64, device="cuda")
        var = torch.empty(m, dtype=torch.float64, device="cuda")
        work = torch.empty((m, N), dtype=torch.float64, device="cuda")
        second = (ptr(Kinv), N) if name == "gprb_predict" else (ptr(Ld), N)
        _lib.call(name, m, N, ptr(Kd), N + 5, ptr(ad), second[0], second[1], ptr(dd), ptr(mean), ptr(var), ptr(work), stream())
        assert rel_err(mean.cpu().numpy(), Ks @ alpha) <= 1e-12
        assert np.abs(var.cpu().numpy() - want_var).max() <= 1e-11 * prior.max()
    # through the GP API: a batch forced through either route gives the same E / F / sigma
    gp = _model(g)
    strucs = [_atoms(g, g["t%d_pos" % k]) for k in range(3)]
    out = {}
    for route in ("inverse", "chol"):
        monkeypatch.setenv("GPRB_VARIANCE_ROUTE", route)
        out[route] = gp.predict_structures(strucs, return_std=True, f_tol=1e-10, batch=3)
    bound = std_tolerance(g["K_b"], 0.002, 0.1, 3, np.array([4.0]))       # on the variance (test_oracle_golden.py)
    for a, b in zip(out["inverse"], out["chol"]):
        assert abs(a[0] - b[0]) <= 1e-10 and np.abs(a[1] - b[1]).max() <= 1e-10
        assert np.abs(np.concatenate(([a[3]], a[4].ravel())) ** 2 - np.concatenate(([b[3]], b[4].ravel())) ** 2).max() <= bound


def test_sparsify_removes_duplicated_points(g):
    """CUR sparsification on device (gaussianprocess.py:1004-1023, 1165-1182): an exactly duplicated training
    structure puts K's smallest eigenvalues below the tolerance and its rows are dropped."""
    from gpr_calculator_b200.gaussianprocess import GP, CUR, CUR_device
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.utilities import convert_train_data
    import torch
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    lab = [(_atoms(g, g["t%d_pos" % k], fixed=False), float(g["t%d_E" % k]), g["t%d_F" % k]) for k in (0, 1, 0)]   # third = first
    gp = GP(kernel=RBF_mb(para=[2.0, 0.8], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(TrainData=convert_train_data(lab, des), opt=False, show=False)
        n_e, n_f = gp.N_energy, gp.N_forces
        K = gp.kernel.k_total(gp.train_x)
        # device and host selections agree
        sel_h = CUR(K[:n_e, :n_e], 1e-8)
        sel_d = CUR_device(torch.as_tensor(K[:n_e, :n_e], device="cuda"), 1e-8)
        # rows 0 and 2 are identical: equal leverage, either may be picked
        assert len(sel_h) == 1 and len(sel_d) == 1 and sel_h[0] in (0, 2) and sel_d[0] in (0, 2)
        gp.sparsify(e_tol=1e-8, f_tol=1e-8)
    # a force centre goes only when all three of its rows are selected; with exact duplicates the selected rows
    # scatter over both copies (ties), so between 1 and 13 centres are dropped (same rule as the reference)
    n_f2 = len(gp.train_x["force"][-1])
    assert len(gp.train_x["energy"][-1]) == n_e - 1 and n_f - 13 <= n_f2 < n_f
    assert len(gp.y_train) == (n_e - 1) + 3 * n_f2 and gp.alpha_ is not None


def _sigma_reference_formula(Kn, Ks, prior):
    """The reference's arithmetic for the predictive standard deviation on a given noisy training matrix
    (gaussianprocess.py:128-131 set_K_inv, 904-908): L = cholesky, L_inv = solve_triangular(L.T, I),
    K_inv = L_inv L_inv^T, var = diag - einsum(K* K_inv, K*), negatives clipped."""
    from scipy.linalg import cholesky, solve_triangular
    L = cholesky(Kn, lower=True)
    L_inv = solve_triangular(L.T, np.eye(len(L)))
    K_inv = L_inv.dot(L_inv.T)
    var = prior - np.einsum("ij,ij->i", np.dot(Ks, K_inv), Ks)
    return np.sqrt(np.maximum(var, 0.0)), L


def _sigma_refined(L, Kn, Ks, prior, sweeps=3):
    """A near-exact value of the same quantity: K z = k* by the Cholesky factor with iterative refinement whose residuals are
    accumulated in extended precision; var = diag - k* . z."""
    from scipy.linalg import cho_solve
    Kl, Kt = Kn.astype(np.longdouble), Ks.T.astype(np.longdouble)
    Z = cho_solve((L, True), Ks.T).astype(np.longdouble)
    for _ in range(sweeps):
        R = Kt - Kl @ Z
        Z = Z + cho_solve((L, True), R.astype(np.float64)).astype(np.longdouble)
    var = prior.astype(np.longdouble) - np.einsum("ji,ji->i", Kt, Z)
    return np.sqrt(np.maximum(var, 0.0)).astype(np.float64)


@pytest.mark.timeout(900)
def test_sigma_routes_against_reference_formula(monkeypatch, capsys):
    """Pins sigma of both device variance routes in the benchmark's regime (real Cu32 rows, l = 0.1, noise 0.002 / 0.1,
    N = 24 + 2 304 = 2 328): against the reference's own formula evaluated in numpy / LAPACK on the same K, and against an
    iteratively refined value.  Tolerances are what each route meets here (printed; recorded in
    profiles/r02_sigma_routes.txt).  Outcome: the factor route is exact to rounding and closer to the reference's numbers
    than a second implementation of the reference's explicit-inverse formula is, so it is the batch route (GP._mean_var)."""
    import torch
    from gpr_calculator_b200 import synthetic as syn, device as gdev
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.batch import rows_from_batch
    des = SO3(nmax=3, lmax=4, rcut=5.0)
    labelled = syn.structures(24, 2, 2000)
    E_dev, F_dev = syn.packed_from_batch(des, [a for a, _, _ in labelled])
    gp = GP(kernel=RBF_mb(para=[1.0, 0.1], zeta=2.0), descriptor=des, noise_e=0.002, noise_f=0.1, log_file=None)
    gp.train_x = {"energy": gdev.Pack(E_dev[0], E_dev[1], E_dev[2]), "force": gdev.Pack(F_dev[0], F_dev[2], F_dev[3], dxdr=F_dev[1])}
    y = syn.targets(labelled)
    gp.train_y = {"energy": list(y[:24, 0]), "force": y[24:, 0].reshape(-1, 3)}
    gp.N_energy, gp.N_forces = 24, 24 * 32
    gp.fit(opt=False, show=False)
    tests_ = [a for a, _, _ in syn.structures(20, 2, 3000)]          # 20 x 97 = 1 940 rows of K*: the batch routes apply
    E_t, F_t = rows_from_batch(des.calculate_batch(tests_, to_host=False), None)
    X = {"energy": gdev.energy_pack(E_t), "force": gdev.force_pack(F_t)}
    Ks, _ = gp.kernel.k_total_device(X, gp.train_x, f_tol=1e-12, grad=False)
    prior = gp.kernel.diag_device(X)
    Kn, _ = gp.kernel.k_total_device(gp.train_x, None, f_tol=1e-10, grad=False)
    Kn = Kn.cpu().numpy()
    idx = np.arange(len(Kn))
    Kn[idx, idx] += np.where(idx < 24, 0.002 ** 2, 0.1 ** 2)
    Ks_h, prior_h = Ks.cpu().numpy(), prior.cpu().numpy()
    sub = np.arange(0, Ks_h.shape[0], 8)             # the extended-precision refinement is slow: every 8th row of K*
    sig_ref, L = _sigma_reference_formula(Kn, Ks_h, prior_h)
    sig_ref = sig_ref[sub]
    sig_true = _sigma_refined(L, Kn, Ks_h[sub], prior_h[sub])
    got = {}
    for route in ("inverse", "chol"):
        monkeypatch.setenv("GPRB_VARIANCE_ROUTE", route)
        _, var = gp._mean_var(Ks, prior)
        got[route] = np.sqrt(var.cpu().numpy())[sub]
    monkeypatch.delenv("GPRB_VARIANCE_ROUTE")
    probe = gp.variance_route_probe(Ks, prior)
    d = {"reference formula vs refined": np.abs(sig_ref - sig_true).max(),
         "device inverse route vs reference formula": np.abs(got["inverse"] - sig_ref).max(),
         "device chol route vs reference formula": np.abs(got["chol"] - sig_ref).max(),
         "device inverse route vs refined": np.abs(got["inverse"] - sig_true).max(),
         "device chol route vs refined": np.abs(got["chol"] - sig_true).max(),
         "device chol vs device inverse": np.abs(got["chol"] - got["inverse"]).max()}
    with capsys.disabled():
        print("\n[sigma routes] N = %d, m = %d, cond(K) = %.3g, sigma range %.3g .. %.3g, probe (first 128 rows) %.3g"
              % (len(Kn), len(sig_ref), np.linalg.cond(Kn), sig_true.min(), sig_true.max(), probe))
        for k, v in d.items():
            print("[sigma routes]   max |d sigma|  %-44s %.3e" % (k, v))
    # pinned tolerances (what each route meets in this regime):
    #   the factor route reproduces the refined value to rounding: 1e-8 in sigma with four orders of margin
    assert d["device chol route vs refined"] <= 1e-10
    #   the reference's own formula is only `floor` away from the refined value: no implementation of that formula can be
    #   asked for more, and the factor route is as close to the reference's numbers as the reference is to the truth
    floor = max(1e-8, 4.0 * d["reference formula vs refined"])
    assert d["device inverse route vs reference formula"] <= floor
    assert d["device chol route vs reference formula"] <= 1.01 * d["reference formula vs refined"] + 1e-10
    assert probe <= 2.0 * floor


@pytest.fixture(scope="module")
def gsel():
    return np.load(os.path.join(GOLD, "selection.npz"))


def _fitted_b(g):
    gp = _model(g)
    gp.kernel.update([2.0, 0.8])
    with contextlib.redirect_stdout(io.StringIO()):
        gp.fit(opt=False, show=False)
    return gp


def test_add_structure_selection_vs_reference(g, gsel):
    """GP.add_structure (gaussianprocess.py:921-1002) against the reference's own run on the same inputs: WHICH force
    centres enter the training set and in what order (incl. the flat-F indexing of :979), the error tuple it returns,
    the queue counters and the appended targets."""
    new = _atoms(g, gsel["new_pos"], fixed=False)
    E_new, F_new = float(gsel["new_E"]), gsel["new_F"]
    cases = {"default": {}, "tight": {"tol_f_var": 0.05}, "capped": {"tol_f_var": 0.05, "N_max": 2}, "noforce": {"add_force": False}}
    for tag, kw in cases.items():
        gp = _fitted_b(g)
        with contextlib.redirect_stdout(io.StringIO()):
            pts, n_pts, err = gp.add_structure((new.copy(), E_new, F_new.copy()), **kw)
        assert list(gp.train_db[-1][4]) == list(gsel[tag + "_force_in"]), tag
        assert n_pts == int(gsel[tag + "_n_pts"])
        assert [gp.N_energy, gp.N_forces, gp.N_energy_queue, gp.N_forces_queue, gp.N_queue] == list(gsel[tag + "_counters"])
        assert np.abs(np.array([err[0], err[1]]) - gsel[tag + "_err_E"][:2]).max() <= 1e-8
        assert np.abs(np.asarray(err[3]) - gsel[tag + "_err_F"]).max() <= 1e-8 and np.abs(np.asarray(err[4]) - gsel[tag + "_err_F1"]).max() <= 1e-8
        assert abs(err[2] - gsel[tag + "_err_E"][2]) <= 1e-6 and np.abs(np.asarray(err[5]) - gsel[tag + "_err_Fstd"]).max() <= 1e-6
        assert np.abs(gp.y_train - gsel[tag + "_y_train"]).max() <= 1e-12
    # untrained model: every centre is a candidate, new_pt() removes near-duplicates
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    from gpr_calculator_b200.SO3 import SO3
    gp = GP(kernel=RBF_mb(para=[2.0, 0.8], zeta=2.0), descriptor=SO3(nmax=3, lmax=4, rcut=5.0), noise_e=0.002, noise_f=0.1, log_file=None)
    with contextlib.redirect_stdout(io.StringIO()):
        for k in range(3):
            gp.add_structure((_atoms(g, g["t%d_pos" % k]), float(g["t%d_E" % k]), g["t%d_F" % k].copy()))
            assert list(gp.train_db[-1][4]) == list(gsel["fresh%d_force_in" % k])
    assert [gp.N_energy, gp.N_forces, gp.N_energy_queue, gp.N_forces_queue, gp.N_queue] == list(gsel["fresh_counters"])


def test_predict_return_cov_vs_reference(g, gsel):
    """GP.predict(X, return_cov=True) (gaussianprocess.py:363-366) on packed test data."""
    from gpr_calculator_b200.SO3 import SO3
    from gpr_calculator_b200.utilities import convert_train_data, list_to_tuple
    gp = _fitted_b(g)
    new = _atoms(g, gsel["new_pos"], fixed=False)
    d = convert_train_data([(new, float(gsel["new_E"]), gsel["new_F"].copy())], SO3(nmax=3, lmax=4, rcut=5.0))
    X = {"energy": list_to_tuple([(d["energy"][0][0], d["energy"][0][2])], mode="energy"),
         "force": list_to_tuple([(f[0], f[1], f[3]) for f in d["force"][9:12]])}
    y_mean, y_cov = gp.predict(X, return_cov=True)
    assert np.abs(y_mean - gsel["cov_mean"]).max() <= 1e-8
    assert y_cov.shape == gsel["cov_cov"].shape and np.abs(y_cov - gsel["cov_cov"]).max() <= 1e-7 * np.abs(gsel["cov_cov"]).max()


def test_cur_selection_vs_reference(gsel):
    """CUR (gaussianprocess.py:1165-1182) on covariance blocks with exactly duplicated training points: the number of
    selected rows, the leverage scores (the projector diagonal onto the low eigen-space) and, where the scores are not tied,
    the selected rows themselves, against the reference's own run."""
    import torch
    from gpr_calculator_b200.gaussianprocess import CUR_device
    K, n_e = gsel["cur_K"], int(gsel["cur_n_e"])
    for tol in (1e-8, 1e-4):
        sel_e = CUR_device(torch.as_tensor(K[:n_e, :n_e], device="cuda"), tol)
        sel_f = CUR_device(torch.as_tensor(K[n_e:, n_e:], device="cuda"), tol)
        ref_e, ref_f, omega = gsel["cur_e_%g" % tol], gsel["cur_f_%g" % tol], gsel["cur_f_omega_%g" % tol]
        assert len(sel_e) == len(ref_e) and len(sel_f) == len(ref_f)
        # rows whose leverage is separated from the cut by more than rounding must agree exactly; ties (exact duplicates have
        # equal leverage in both copies) may be resolved either way by the eigen-solver
        cut = np.sort(omega)[::-1][len(ref_f) - 1] if len(ref_f) else 0.0
        sure = set(np.flatnonzero(omega > cut + 1e-6))
        assert sure <= set(int(i) for i in sel_f) and sure <= set(int(i) for i in ref_f)
        assert np.all(omega[sel_f] >= cut - 1e-6)


def test_blocked_cholesky_single_rank():
    """dist.distributed_cholesky on one rank is a plain right-looking blocked Cholesky (gprb_chol_panel + gprb_chol_trailing):
    factor against scipy, ragged last panel, and the status of a matrix that is not positive definite."""
    import torch
    from scipy.linalg import cholesky
    from gpr_calculator_b200 import dist as gdist
    rng = np.random.default_rng(31)
    for N, nb in ((700, 128), (513, 512), (96, 1024)):
        A = rng.normal(size=(N, N))
        K = A @ A.T + N * np.eye(N)
        Kd = torch.as_tensor(K, device="cuda").contiguous()
        assert gdist.distributed_cholesky(Kd, nb=nb) == 0
        L = np.tril(Kd.cpu().numpy())
        assert rel_err(L, cholesky(K, lower=True)) <= 1e-12 and rel_err(L @ L.T, K) <= 1e-13
    A = rng.normal(size=(700, 700))
    K = A @ A.T + 700 * np.eye(700)
    K[300, 300] = -1.0
    assert gdist.distributed_cholesky(torch.as_tensor(K, device="cuda").contiguous(), nb=128) > 0
