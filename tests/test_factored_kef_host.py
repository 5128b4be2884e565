"""CPU: the factored K_fe / K_ef algebra (DESIGN.md §2) and its DMMA counts (csrc/cov_factored.cu).

* A numpy restatement of K_fe(3J+c, I) = -(1/n_I) sum_k A~_c(J,k) . Y_I(k), Y_I(k) = sum_{a in I} W1(a,k) x^(a), against
  the oracle's pairwise K_ef and dK_ef/dl on the force rows of test_factored_kff_host.shared_atom_data (three species, a
  dropped atom, duplicate rows in a group).
* gprb_atom_plan_cost_kef at the S5 and S4 shapes and at one centre per structure."""
import ctypes

import numpy as np
import pytest

from helpers import rel_err
from test_factored_kff_host import shared_atom_data


def _unit(x):
    n = np.linalg.norm(x, axis=1)
    keep = n > 1e-8
    return np.where(keep[:, None], x / np.where(keep, n, 1.0)[:, None], 0.0), keep


def factored_kef(structs, items, energy, sigma, l, zeta):
    """K_ef and dK_ef/dl (RBF, [NE, 3 NF]) through the sums regrouped over each structure's atoms."""
    c = 1.0 / (2 * l * l)
    k1 = sigma ** 2 * c
    NE, NF = len(energy), len(items)
    K = np.zeros((NE, 3 * NF))
    dK = np.zeros((NE, 3 * NF))
    for J, (s, atoms, dx) in enumerate(items):
        xT, zT = structs[s]
        xhT, keepT = _unit(xT)
        A = np.zeros((xT.shape[0], xT.shape[1], 3))           # A~ summed per atom of the group
        x = xT[atoms]
        n = np.linalg.norm(x, axis=1)
        for r, j in enumerate(atoms):
            if n[r] <= 1e-8:
                continue
            h = x[r] / n[r]
            A[j] += (dx[r] - np.outer(h, h @ dx[r])) / n[r]
        for I, (xI, zI) in enumerate(energy):
            xhI, keepI = _unit(xI)
            s_ = xhI @ xhT.T                                   # [a, k]
            valid = (zI[:, None] == zT[None, :]) & keepI[:, None] & keepT[None, :]
            sv = np.where(valid, s_, 1.0)
            D = sv ** zeta
            W1 = np.exp(-(1 - D) * c) * k1 * zeta * sv ** (zeta - 1)
            U1 = W1 * ((1 - D) / l ** 3 - 2 / l)
            for W, out in ((W1, K), (U1, dK)):
                Y = np.einsum('ak,ad->kd', np.where(valid, W, 0.0), xhI)
                out[I, 3 * J:3 * J + 3] = -np.einsum('kdc,kd->c', A, Y) / xI.shape[0]
    return K, dK


def test_regrouped_kef_matches_pairwise_oracle(oracle_libs):
    ok = oracle_libs
    rng = np.random.default_rng(7)
    structs, items = shared_atom_data(rng)
    # energy groups: every structure (one with a dropped atom), and one group mixing atoms of two structures
    energy = [(x, z) for x, z in structs]
    energy.append((np.concatenate([structs[0][0][:3], structs[2][0][2:6]]),
                   np.concatenate([structs[0][1][:3], structs[2][1][2:6]])))
    F = ok.list_to_tuple([(structs[s][0][atoms], dx, structs[s][1][atoms]) for s, atoms, dx in items])
    E = ok.list_to_tuple(energy, mode="energy")
    O = ok.RBFOracle("port")
    for zeta in (2.0, 3.0):
        K_ref, _, dK_ref = O.kef_C(E, F, 1.3, 0.7, zeta, grad=True)
        K, dK = factored_kef(structs, items, energy, 1.3, 0.7, zeta)
        assert np.abs(K_ref).max() > 0 and np.abs(dK_ref).max() > 0
        assert rel_err(K, K_ref) <= 1e-13
        assert rel_err(dK, dK_ref) <= 1e-13


def _cost_kef(cg, cs, n_rows, ne_rows, ne):
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    pw, fa = ctypes.c_double(), ctypes.c_double()
    cg = np.ascontiguousarray(cg, np.int32)
    cs = np.ascontiguousarray(cs, np.int32)
    assert lib.gprb_atom_plan_cost_kef(len(cs), cg.ctypes.data, cs.ctypes.data, n_rows, ne_rows, ne,
                                       ctypes.byref(pw), ctypes.byref(fa)) == 0
    return pw.value, fa.value


@pytest.mark.parametrize("n_atoms, rows", [(32, 29), (108, 100)])
def test_kef_cost_model_s5_s4_shapes(n_atoms, rows):
    # 340 x Cu32 (S5) and 200 x Cu108 (S4): one energy group per structure, one force centre per atom
    n_struct = 340 if n_atoms == 32 else 200
    cg = np.arange(0, n_atoms * (n_struct + 1), n_atoms)
    cs = np.full(n_struct, n_atoms)
    n_rows, ne_rows = n_struct * n_atoms * rows, n_struct * n_atoms
    pw, fa = _cost_kef(cg, cs, n_rows, ne_rows, n_struct)
    npad = (n_atoms + 7) // 8 * 8
    etiles = (ne_rows + 7) // 8
    assert pw == 32 * ((n_rows + 7) // 8) * etiles
    assert fa == n_struct * (24 * etiles * npad // 8 + -(-3 * n_atoms // 8) * -(-2 * n_struct // 8) * 8 * npad)
    assert pw >= 10 * fa


def test_kef_one_centre_per_structure_keeps_the_pairwise_kernel():
    # the add_structure regime: every force group is a cluster of its own
    rng = np.random.default_rng(1)
    sizes = rng.integers(20, 33, size=200)
    cg = np.concatenate(([0], np.arange(1, 201)))
    pw, fa = _cost_kef(cg, sizes, int(sizes.sum()), int(sizes.sum()), 200)
    assert pw < 2 * fa
