"""CPU: host-side logic of the drop-in (layouts, block assembly, selection, sharding, bookkeeping)."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from helpers import make_force, make_energy


def test_list_tuple_roundtrip():
    from gpr_calculator_b200.utilities import list_to_tuple, tuple_to_list
    rng = np.random.default_rng(0)
    fl = make_force(rng, 5, lo=1, hi=6)
    X, dX, ELE, ind = list_to_tuple(fl)
    assert X.shape[0] == sum(ind) == dX.shape[0] == len(ELE) and dX.shape[2] == 3
    back = tuple_to_list((X, dX, ELE, ind))
    for (x, dx, e), (x2, dx2, e2) in zip(fl, back):
        assert np.array_equal(x, x2) and np.array_equal(dx, dx2) and np.array_equal(e, e2)
    el = make_energy(rng, 3)
    Xe, Ee, inde = list_to_tuple(el, mode="energy")
    assert [len(x) for x, _ in el] == inde
    with_vals = list_to_tuple([(x, dx, np.ones(3) * i, e) for i, (x, dx, e) in enumerate(fl)], include_value=True)
    assert len(with_vals) == 5 and len(with_vals[4]) == 5


def test_list_to_tuple_matches_oracle_layout():
    from gpr_calculator_b200.utilities import list_to_tuple
    from oracle.kernels import list_to_tuple as olt
    rng = np.random.default_rng(1)
    fl = make_force(rng, 4)
    for a, b in zip(list_to_tuple(fl), olt(fl)):
        assert np.array_equal(np.asarray(a), np.asarray(b))


def test_build_covariance_dispatch():
    from gpr_calculator_b200.kernels.base import build_covariance
    ee, ef, fe, ff = np.ones((2, 2)), 2 * np.ones((2, 6)), 3 * np.ones((6, 2)), 4 * np.ones((6, 6))
    assert build_covariance(ee, ef, fe, ff).shape == (8, 8)
    assert build_covariance(None, None, fe, ff).shape == (6, 8)
    assert build_covariance(ee, ef, None, None).shape == (2, 8)
    assert build_covariance(None, ef, None, None) is ef
    assert build_covariance(None, None, None, ff) is ff
    assert build_covariance(ee, None, fe, None) is None      # not in the reference's table either


def test_new_pt():
    from gpr_calculator_b200.utilities import new_pt
    x = np.array([1.0, 2.0, 3.0])
    assert not new_pt((x, 29), [(x * 1.01, 29)])
    assert new_pt((x, 29), [(x * 1.01, 13)])
    assert new_pt((x, 29), [(np.array([3.0, -1.0, 0.1]), 29)])


def test_split_groups_and_windows():
    from gpr_calculator_b200.dist import split_groups, row_windows, window_row_ranges
    rng = np.random.default_rng(2)
    costs = rng.integers(20, 40, size=101)
    for parts in (1, 2, 3, 4, 8):
        b = split_groups(costs, parts)
        assert b[0] == 0 and b[-1] == len(costs) and all(b[i] <= b[i + 1] for i in range(parts))
        loads = [costs[b[i]:b[i + 1]].sum() for i in range(parts)]
        assert max(loads) - min(loads) <= 2 * costs.max()
    assert split_groups([], 4) == [0, 0, 0, 0, 0]
    w = row_windows([32] * 5, [30] * 17, 4)
    rr = window_row_ranges(w, NE=5)
    covered = sorted(r for pair in rr for r in pair)
    # energy windows tile [0,5), force windows tile [5, 5+51)
    assert covered[0][0] == 0 and max(hi for _, hi in covered) == 5 + 3 * 17


def _toy_gp():
    from gpr_calculator_b200.gaussianprocess import GP
    from gpr_calculator_b200.kernels import RBF_mb
    return GP(kernel=RBF_mb(para=[1.0, 0.1]), descriptor=None, log_file=None)


def test_gp_bookkeeping_without_gpu():
    rng = np.random.default_rng(3)
    gp = _toy_gp()
    fl = make_force(rng, 4, lo=2, hi=5)
    el = make_energy(rng, 2, lo=3, hi=6)
    data = {"energy": [(x, 0.5 * i, e) for i, (x, e) in enumerate(el)],
            "force": [(x, dx, np.full(3, float(i)), e) for i, (x, dx, e) in enumerate(fl)],
            "db": [("s0", 1.0, None, True, [0, 1]), ("s1", 2.0, None, True, [0, 1])]}
    gp.set_train_pts(data)
    assert (gp.N_energy, gp.N_forces, gp.N_queue) == (2, 4, 6)
    assert gp.y_train.shape == (2 + 12, 1)
    assert np.array_equal(gp.y_train[:, 0], [0.0, 0.5] + [0.0] * 3 + [1.0] * 3 + [2.0] * 3 + [3.0] * 3)
    # queue slicing: pretend the first energy and two forces are fitted
    gp.N_energy_queue, gp.N_forces_queue, gp.N_queue = 1, 2, 3
    tx = gp.get_train_x()
    assert len(tx["energy"][-1]) == 1 and len(tx["force"][-1]) == 2
    assert tx["force"][0].shape[0] == sum(tx["force"][-1])
    # append mode
    gp.set_train_pts({"energy": data["energy"][:1], "force": data["force"][:1], "db": [("s2", 0.0, None, True, [0])]}, mode="a+")
    assert (gp.N_energy, gp.N_forces) == (3, 5) and gp.y_train.shape[0] == 3 + 15
    assert "RBF" in str(gp) and "3 energy" in str(gp)


def test_so3_validation_and_dict():
    from gpr_calculator_b200.SO3 import SO3
    s = SO3(nmax=3, lmax=4, rcut=5.0)
    assert s.ncoefs == 30
    d = s.save_dict()
    assert d["_type"] == "SO3" and d["lmax"] == 4
    t = SO3()
    t.load_from_dict(d)
    assert (t.nmax, t.lmax, t.rcut) == (3, 4, 5.0)
    for bad in (dict(nmax=0), dict(nmax=12), dict(nmax=2.5), dict(lmax=-1), dict(rcut=-1.0), dict(alpha=0), dict(derivative=1)):
        with pytest.raises(ValueError):
            SO3(**bad)
    with pytest.raises(NotImplementedError):
        SO3(cutoff_function="tanh")


def test_kernel_object_surface():
    from gpr_calculator_b200.kernels import RBF_mb, Dot_mb
    k = RBF_mb(para=[2.0, 0.5], zeta=2)
    assert str(k) == "2.00000**2 *RBF(0.50000)" and k.parameters() == [2.0, 0.5] and k.name == "RBF"
    k2 = RBF_mb()
    k2.load_from_dict(k.save_dict())
    assert k2.parameters() == [2.0, 0.5] and k2.bounds == [[1e-2, 5e+1], [1e-1, 1e+1]]
    d = Dot_mb(para=[2, 2.0], zeta=3)
    assert str(d) == "2.000**2 *Dot(2.000)" and d.save_dict()["sigma0"] == 2.0


def test_cur_selects_null_space_rows():
    from gpr_calculator_b200.gaussianprocess import CUR
    v = np.array([1.0, 1.0, 0.0])
    K = np.outer(v, v) + np.diag([0.0, 0.0, 1.0])     # rows 0 and 1 are redundant
    ids = CUR(K, 1e-10)
    assert len(ids) == 1 and ids[0] in (0, 1)


def test_gpr_adapter_gate_and_refit_cadence(capsys):
    """GPR.calculate control flow with a scripted surrogate (no GPU): uncertainty gate
    (calculator.py:62-73), base fall-back + add_structure, refit trigger (:101-103), freeze()."""
    import numpy as np
    from gpr_calculator_b200.calculator import GPR
    from gpr_calculator_b200.utilities import SimpleAtoms, FixAtoms

    class FakeGP:
        noise_e, noise_f = 0.002, 0.1
        use_base = use_surrogate = fits = 0
        N_forces = N_queue = N_energy_queue = 0
        error = {"energy_mae": 0.0, "forces_mae": 0.0}
        f_std = 0.01

        def predict_structure(self, atoms, stress, return_std, f_tol=1e-12):
            n = len(atoms)
            return 1.0, np.full((n, 3), 0.05), None, 0.001, np.full((n, 3), self.f_std)

        def add_structure(self, data):
            self.N_queue += 3
            self.N_energy_queue += 1

        def fit(self, opt=True, show=False, maxiter=10):
            self.fits += 1
            self.N_queue = self.N_energy_queue = 0

        def validate_data(self, show=False):
            pass

    class Base:
        def get_potential_energy(self, atoms):
            return -7.0

        def get_forces(self, atoms):
            return np.ones((len(atoms), 3))

    at = SimpleAtoms([13, 13, 79], np.zeros((3, 3)), np.eye(3) * 5, constraints=[FixAtoms([0])])
    gp = FakeGP()
    calc = GPR(base=Base(), ff=gp, save=False, freq=10)
    calc.calculate(at)                                    # F_std 0.01 < max(0.12, 0.05/2.5): surrogate
    assert gp.use_surrogate == 1 and gp.use_base == 0 and calc.results["energy"] == 1.0
    gp.f_std = 0.5                                        # above the gate: base calculator, labels replace the prediction
    calc.calculate(at)
    assert gp.use_base == 1 and calc.results["energy"] == -7.0
    assert np.all(calc.results["forces"][0] == 0.0) and np.all(calc.results["forces"][1:] == 1.0)   # FixAtoms rows zeroed
    assert gp.fits == 0 and gp.N_energy_queue == 1
    calc.calculate(at)                                    # second queued energy triggers the refit (N_energy_queue >= 2)
    assert gp.use_base == 2 and gp.fits == 1 and gp.N_queue == 0
    calc.freeze()
    calc.calculate(at)
    assert gp.use_base == 2 and gp.use_surrogate == 2     # frozen: never calls the base
    out = capsys.readouterr().out
    assert out.count("From Base model") == 2 and out.count("From Surrogate") == 2
    assert calc.get_var_f().shape == (3, 3) and calc.get_e() == calc.results["energy"] / 3


def test_synthetic_pair_counts_and_windows():
    import numpy as np
    from gpr_calculator_b200.synthetic import pair_counts, cu_fcc
    from gpr_calculator_b200 import dist as gd
    ele = np.array([29] * 5 + [13] * 3 + [29] * 2)
    ind = [4, 4, 2]                                       # groups: 4x29 | 29,13,13,13 | 29,29
    full = pair_counts(ele, ind, symmetric=False)
    assert full == 7 * 7 + 3 * 3
    up = pair_counts(ele, ind, symmetric=True)
    brute = sum((ele[a] == ele[b]) for I in range(3) for J in range(I, 3)
                for a in range(sum(ind[:I]), sum(ind[:I + 1])) for b in range(sum(ind[:J]), sum(ind[:J + 1])))
    assert up == brute
    at, E, F = cu_fcc(2, 7)
    assert len(at) == 32 and F.shape == (32, 3) and E > 0
    w = gd.row_windows([32] * 7, [28] * 40, 4, upper=True)
    sizes = [f1 - f0 for _, (f0, f1) in w]
    assert sum(sizes) == 40 and sizes[0] < sizes[-1]      # early rows carry longer sweeps


def test_row_pieces_cover_rows_once():
    """Blocks of the inverse-rows likelihood gradient: every held row exactly once, never across the energy / force
    boundary, dK offsets consecutive."""
    from gpr_calculator_b200.gaussianprocess import _row_pieces
    for NE, N, ranges in ((340, 32980, [(0, 32980)]), (0, 900, [(0, 900)]), (5, 5, [(0, 5)]), (7, 100, [(2, 5), (40, 73)]),
                          (7, 100, [(0, 7), (7, 100)]), (340, 32980, [(170, 340), (20000, 32980)]), (3, 50, [(0, 0), (3, 3)])):
        pieces = _row_pieces(ranges, NE, N, parts=16, min_rows=4)
        rows, off = [], 0
        for (a, b, doff) in pieces:
            assert b > a and (b <= NE or a >= NE)
            assert doff == off
            off += b - a
            rows += list(range(a, b))
        want = [i for (r0, r1) in ranges for i in range(r0, r1)]
        assert rows == want


def test_trailing_block_inverse_identity():
    """K^-1[T, T] = (L_TT L_TT^T)^-1 for a trailing index set T (what gprb_chol_inverse_rows relies on)."""
    rng = np.random.default_rng(5)
    A = rng.normal(size=(40, 40))
    K = A @ A.T + 40 * np.eye(40)
    L = np.linalg.cholesky(K)
    Kinv = np.linalg.inv(K)
    for c0 in (0, 7, 33):
        LT = L[c0:, c0:]
        assert np.allclose(np.linalg.inv(LT @ LT.T), Kinv[c0:, c0:], rtol=1e-10, atol=1e-12)


def test_zero_build_targets_and_slab_pointers():
    import torch
    from gpr_calculator_b200.gaussianprocess import _zero_build_targets
    from gpr_calculator_b200.dist import slab_pointers
    NE, NF = 3, 11
    N = NE + 3 * NF
    K = torch.ones((N, N), dtype=torch.float64)
    _zero_build_targets(K, NE, chunks=4)
    i, j = np.indices((N, N))
    must_zero = (i >= NE) & ((j < NE) | (j >= i))           # K_fe columns and the F-F part on / right of the diagonal
    assert bool((K.numpy()[must_zero] == 0).all())
    assert bool((K.numpy()[:NE] == 1).all())                # energy rows untouched
    assert slab_pointers([1000, 5000], 4, 2, 10) == [1000 + (4 * 10 + 2) * 8, 5000 + (4 * 10 + 2) * 8]


def _check_get_data(des, tol):
    """utilities.get_data / get_strucs / get_train_data / convert_struc against the reference's own output on the
    committed 3-row database (tests/golden/gen_golden_getdata.py)."""
    import os
    from gpr_calculator_b200 import utilities as ut
    gold = os.path.join(os.path.dirname(__file__), "golden")
    g = np.load(os.path.join(gold, "getdata.npz"))
    db = os.path.join(gold, "getdata.db")
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        cases = {"all": ut.get_data(db, des), "cap": ut.get_data(db, des, N_force=17),
                 "sel": ut.get_data(db, des, lists=[0, 2], select=True), "noe": ut.get_data(db, des, N_force=5, no_energy=True)}
    for name, data in cases.items():
        assert len(data["energy"]) == int(g[name + "_nE"]) and len(data["force"]) == int(g[name + "_nF"])
        assert [len(x) for x, _, _, _ in data["force"]] == list(g[name + "_F_rows"])
        assert [len(f) for _, _, _, _, f in data["db"]] == list(g[name + "_db_fids"])
        assert np.array_equal(np.array([y for _, _, y, _ in data["force"]]), g[name + "_F_y"])
        Fx = np.concatenate([x for x, _, _, _ in data["force"]])
        Fd = np.concatenate([d for _, d, _, _ in data["force"]])
        if name == "all":
            assert abs(np.abs(Fx).sum() - g["all_F_x_abs_sum"]) <= tol * g["all_F_x_abs_sum"]
            assert abs(np.abs(Fd).sum() - g["all_F_dxdr_abs_sum"]) <= tol * g["all_F_dxdr_abs_sum"]
            continue
        assert np.abs(Fx - g[name + "_F_x"]).max() <= tol * np.abs(g[name + "_F_x"]).max()
        assert np.abs(Fd - g[name + "_F_dxdr"]).max() <= tol * np.abs(g[name + "_F_dxdr"]).max()
        assert np.array_equal(np.concatenate([e for _, _, _, e in data["force"]]), g[name + "_F_ele"])
        assert np.array_equal(np.array([E for _, E, _, _, _ in data["db"]]), g[name + "_db_E"])
        if data["energy"]:
            Ex = np.concatenate([x for x, _, _ in data["energy"]])
            assert np.abs(Ex - g[name + "_E_x"]).max() <= tol * np.abs(g[name + "_E_x"]).max()
            assert np.array_equal(np.array([y for _, y, _ in data["energy"]]), g[name + "_E_y"])
            assert np.array_equal(np.concatenate([e for _, _, e in data["energy"]]), g[name + "_E_ele"])
    S, V = ut.get_strucs(db, N_max=2)
    assert len(S) == int(g["strucs_n"]) and np.array_equal(np.array([v[0] for v in V]), g["strucs_E"]) and V[0][2] is None
    strucs, energies, forces = ut.get_train_data(db)
    assert len(strucs) == 3 and np.array_equal(np.array(energies)[:2], g["strucs_E"]) and forces[0].shape == (13, 3)
    xs, Y, st = ut.convert_struc(db, des, ids=[1], N=1)
    assert len(xs) == 1 and len(st) == 1 and Y["energy"] == [energies[1]]
    assert "R2" in ut.metric_single(np.arange(5.0), np.arange(5.0) + 0.1, "Energy", show_max=True)
    assert len(ut.metrics(np.arange(5.0), np.arange(3.0), np.arange(5.0), np.arange(3.0), "F")) == 2


def test_get_data_with_oracle_descriptor():
    from oracle import so3 as oso3
    _check_get_data(oso3.SO3Oracle(3, 4, 5.0, 2.0), 1e-10)


def test_inverse_rows_gradient_algebra_in_numpy():
    """The blocked route of GP._lml_gradient_rows restated in numpy: 1/2 tr((alpha alpha^T - K^-1) dK) from trailing-block
    solves only (K^-1[r0:r1, r0:] per block, K^-1[0:NE, :] for the energy columns), with the sharded-row semantics of the
    trace kernel (energy rows: E-E part on / right of the diagonal doubled; force rows: 2 x F-E + F-F on / right of the
    diagonal doubled), equals the dense formula of gaussianprocess.py:188-198."""
    from scipy.linalg import solve_triangular
    from gpr_calculator_b200.gaussianprocess import _row_pieces
    rng = np.random.default_rng(12)
    NE, N = 5, 61
    A = rng.normal(size=(N, N))
    K = A @ A.T + N * np.eye(N)
    B = rng.normal(size=(N, N))
    dK = B + B.T
    alpha = rng.normal(size=N)
    W = np.outer(alpha, alpha) - np.linalg.inv(K)
    want = 0.5 * np.sum(W * dK)
    L = np.linalg.cholesky(K)

    def inverse_rows(r0, r1, c0):
        LT = L[c0:, c0:]
        E = np.zeros((N - c0, r1 - r0))
        E[np.arange(r0 - c0, r1 - c0), np.arange(r1 - r0)] = 1.0
        Y = solve_triangular(LT, E, lower=True)
        return solve_triangular(LT.T, Y, lower=False).T              # [r1 - r0, N - c0]

    Einv = inverse_rows(0, NE, 0)
    got = 0.0
    # two "ranks": their row ranges together cover every row once, like dist.row_windows
    for ranges in ([(0, 2), (NE, NE + 21)], [(2, NE), (NE + 21, N)]):
        for (r0, r1, _) in _row_pieces(ranges, NE, N, parts=4, min_rows=4):
            rows = Einv[r0:r1] if r1 <= NE else inverse_rows(r0, r1, r0)
            c0 = 0 if r1 <= NE else r0
            for i in range(r0, r1):
                jend = NE if i < NE else N
                for j in range(i, jend):
                    w = alpha[i] * alpha[j] - rows[i - r0, j - c0]
                    got += (0.5 if j == i else 1.0) * w * dK[i, j]
                if i >= NE:
                    for j in range(NE):
                        got += (alpha[i] * alpha[j] - Einv[j, i]) * dK[i, j]
    assert abs(got - want) <= 1e-10 * abs(want)


def test_gpr_calc_import_alias():
    """The reference's import paths (README.md:34-71) resolve to the B200 modules themselves."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from gpr_calc.gaussianprocess import GP\nfrom gpr_calc.calculator import GPR\n"
            "from gpr_calc.kernels.RBF_mb import RBF_mb\nfrom gpr_calc.kernels.Dot_mb import Dot_mb\nfrom gpr_calc.SO3 import SO3\n"
            "from gpr_calc.utilities import list_to_tuple\nimport gpr_calculator_b200.gaussianprocess as g, gpr_calculator_b200.SO3 as s\n"
            "assert GP is g.GP and SO3 is s.SO3 and RBF_mb(para=[1.0, 0.1]).l == 0.1\nprint('alias ok')\n" % ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "alias ok" in res.stdout, res.stderr[-2000:]


def test_two_stage_contraction_emulation(capsys):
    """The register-level algebra of the default no-gradient K_ff kernel (stage-1 accumulators fed unchanged as stage-2 A fragments,
    stage-2 B fragments read from the production slab layout, a column tile that straddles two groups) against the direct pair
    sums: numpy emulation of the m8n8k4 lane layouts (profiles/experiments/two_stage_emulation.py)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("two_stage_emulation",
                                                  os.path.join(ROOT, "profiles", "experiments", "two_stage_emulation.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.main()                                  # asserts the 3x3 blocks to 1e-12
    assert "two-stage vs direct" in capsys.readouterr().out


def test_lml_eval_workspace_size():
    """Host-only entry point of the C ABI: workspace of gprb_lml_eval = (NE + block of rows) x N doubles, block = max(512, N / parts)."""
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    assert lib.gprb_lml_eval_work(32980, 340, 1, 16) == (340 + 2062) * 32980
    assert lib.gprb_lml_eval_work(172, 4, 1, 16) == (4 + 172) * 172          # one block: the whole matrix
    assert lib.gprb_lml_eval_work(32980, 340, 0, 16) == 0                    # no gradient: nothing to hold


def test_pack_create_rejects_descriptors_longer_than_64():
    """gprb_pack_create refuses d > 64 (no covariance kernel takes it) with GPRB_ERR_UNSUPPORTED before any CUDA call,
    for energy and force packs whose other arguments are all valid."""
    import ctypes
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    rows = np.array([2, 3], dtype=np.int32)
    ele = np.array([1, 1, 8, 8, 8], dtype=np.int32)
    for d in (65, 72):
        x = np.ones((5, d))
        for ncols, dxdr in ((0, None), (3, np.ones((5, d, 3)))):
            out = ctypes.c_void_p(0)
            rc = lib.gprb_pack_create(ctypes.byref(out), 2, rows.ctypes.data, d, ncols, x.ctypes.data,
                                      None if dxdr is None else dxdr.ctypes.data, ele.ctypes.data, 0.0, None)
            assert rc == _lib.ERR_UNSUPPORTED and not out.value, (d, ncols, rc)
