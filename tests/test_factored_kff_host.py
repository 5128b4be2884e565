"""CPU: the factored K_ff algebra (DESIGN.md §2) and the host part of the atom plan (csrc/cov_factored.cu).

* A numpy restatement of K_ce(I,J) = sum_j A~_c(I,j) . Z_e(J,j) against the oracle's pairwise K_ff and dK/dl on
  rows that are copies of a few atoms' descriptors: three species, a dropped (zero) atom, duplicate rows in a group.
* gprb_atom_plan_host / gprb_atom_plan_cost on crafted keys: cluster cuts, collisions, no sharing."""
import ctypes

import numpy as np
import pytest

from helpers import rel_err


def shared_atom_data(rng, n_struct=3, n_atoms=7, n_centres=4, d=30, species=(8, 12, 46)):
    """Per structure: atom descriptors and species; every centre gets rows = neighbour atoms (with a duplicate)."""
    base = np.abs(rng.normal(size=d)) + 0.5
    structs, items = [], []
    for s in range(n_struct):
        x = base[None, :] + 0.3 * rng.normal(size=(n_atoms, d))
        z = rng.choice(species, size=n_atoms)
        if s == 1:
            x[2] = 0.0                                       # a dropped atom (|x| <= eps)
        structs.append((x, z))
        for i in range(n_centres):
            atoms = [j for j in range(n_atoms) if rng.random() < 0.8] or [0]
            atoms.append(atoms[0])                           # the same atom twice in one group
            atoms = np.array(atoms)
            items.append((s, atoms, rng.normal(size=(len(atoms), d, 3))))
    return structs, items


def factored_kff(structs, items, sigma, l, zeta):
    """K_ff and dK/dl (RBF) through the regrouped sums."""
    xh, atil = [], []
    for x, _ in structs:
        n = np.linalg.norm(x, axis=1)
        keep = n > 1e-8
        xh.append(np.where(keep[:, None], x / np.where(keep, n, 1.0)[:, None], 0.0))
    n_atoms = structs[0][0].shape[0]
    for s, atoms, dx in items:
        A = np.zeros((n_atoms, dx.shape[1], 3))               # A~ summed per atom of the group
        x = structs[s][0][atoms]
        n = np.linalg.norm(x, axis=1)
        for r, j in enumerate(atoms):
            if n[r] <= 1e-8:
                continue
            h = x[r] / n[r]
            A[j] += (dx[r] - np.outer(h, h @ dx[r])) / n[r]
        atil.append(A)
    c = 1.0 / (2 * l * l)
    k1 = sigma ** 2 * c
    NF = len(items)
    K = np.zeros((3 * NF, 3 * NF))
    dK = np.zeros((3 * NF, 3 * NF))
    for I, (S, _, _) in enumerate(items):
        for J, (T, _, _) in enumerate(items):
            s = xh[S] @ xh[T].T
            zS, zT = structs[S][1], structs[T][1]
            valid = (zS[:, None] == zT[None, :]) & (np.linalg.norm(xh[S], axis=1)[:, None] > 0) & \
                    (np.linalg.norm(xh[T], axis=1)[None, :] > 0)
            sv = np.where(valid, s, 1.0)
            D = sv ** zeta
            E = np.exp(-(1 - D) * c)
            W1 = E * k1 * zeta * sv ** (zeta - 1)
            q2 = k1 * zeta ** 2 * sv ** (2 * zeta - 2)
            W2 = E * (k1 * zeta * (zeta - 1) * sv ** (zeta - 2) + q2 * c)
            h = (1 - D) / l ** 3 - 2 / l
            U1, U2 = W1 * h, W2 * h - E * q2 / l ** 3
            W1, W2, U1, U2 = (np.where(valid, w, 0.0) for w in (W1, W2, U1, U2))
            B = atil[J]                                       # [k, d, e]
            q = np.einsum('jd,kde->jke', xh[S], B)            # x^(j) . B~_e(J, k)
            for W, V, out in ((W1, W2, K), (U1, U2, dK)):
                Z = np.einsum('jk,kde->jde', W, B) + np.einsum('jk,jke,kd->jde', V, q, xh[T])
                out[3 * I:3 * I + 3, 3 * J:3 * J + 3] = np.einsum('jdc,jde->ce', atil[I], Z)
    return K, dK


def test_regrouped_sums_match_pairwise_oracle(oracle_libs):
    ok = oracle_libs
    rng = np.random.default_rng(7)
    structs, items = shared_atom_data(rng)
    rows = [(structs[s][0][atoms], dx, structs[s][1][atoms]) for s, atoms, dx in items]
    F = ok.list_to_tuple(rows)
    O = ok.RBFOracle("port")
    for zeta in (2.0, 3.0):
        K_ref, _, dK_ref = O.kff_C(F, F, 1.3, 0.7, zeta, grad=True)
        K, dK = factored_kff(structs, items, 1.3, 0.7, zeta)
        assert rel_err(K, K_ref) <= 1e-13
        assert rel_err(dK, dK_ref) <= 1e-13


# ---- host plan ---------------------------------------------------------------------------------------------------

def _plan(group_keys, a_max=128, max_groups=4096, unique=None):
    """group_keys: per group a list of (hash, code) row keys."""
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    sizes = [len(g) for g in group_keys]
    G = len(sizes)
    row_ptr = np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)
    R = int(row_ptr[-1])
    keys = [k for g in group_keys for k in g]
    h = np.array([k[0] for k in keys], dtype=np.uint64)
    c = np.array([k[1] for k in keys], dtype=np.int32)
    u = None if unique is None else np.asarray(unique, dtype=np.uint8)
    nc = ctypes.c_int()
    cg = np.zeros(G + 1, np.int32)
    cs = np.zeros(max(G, 1), np.int32)
    rs = np.zeros(max(R, 1), np.int32)
    rep = np.zeros(max(R, 1), np.int32)
    rc = lib.gprb_atom_plan_host(G, row_ptr.ctypes.data, h.ctypes.data, c.ctypes.data,
                                 None if u is None else u.ctypes.data, a_max, max_groups,
                                 ctypes.byref(nc), cg.ctypes.data, cs.ctypes.data, rs.ctypes.data, rep.ctypes.data)
    n = nc.value
    return rc, n, cg[:n + 1], cs[:n], rs[:R], rep[:max(int(cs[:n].sum()), 0)], row_ptr


def _cost(n, cg, cs, R, upper):
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    pw, fa = ctypes.c_double(), ctypes.c_double()
    cg = np.ascontiguousarray(cg, np.int32)
    cs = np.ascontiguousarray(cs, np.int32)
    assert lib.gprb_atom_plan_cost(n, cg.ctypes.data, cs.ctypes.data, R, int(upper), ctypes.byref(pw), ctypes.byref(fa)) == 0
    return pw.value, fa.value


def _structures(n_struct, n_atoms, rows_per_group, rng):
    groups = []
    for s in range(n_struct):
        for i in range(n_atoms):
            atoms = rng.choice(n_atoms, size=rows_per_group, replace=False)
            groups.append([(1000 * s + int(a) + 1, 29) for a in sorted(atoms)])
    return groups


def test_plan_one_cluster_per_structure_and_slots():
    rng = np.random.default_rng(0)
    groups = _structures(5, 32, 28, rng)
    rc, n, cg, cs, rs, rep, row_ptr = _plan(groups)
    assert rc == 0 and n == 5
    assert list(cg) == [0, 32, 64, 96, 128, 160]
    assert all(cs <= 32)
    keys = [k for g in groups for k in g]
    slot0 = np.concatenate(([0], np.cumsum(cs)))
    for g in range(len(groups)):
        cl = int(np.searchsorted(cg, g, side="right") - 1)
        for r in range(row_ptr[g], row_ptr[g + 1]):
            assert keys[rep[slot0[cl] + rs[r]]] == keys[r]     # every row's slot holds its key
    # S5-like shapes take the factored path (>= 2x fewer DMMAs), in both modes
    for upper in (True, False):
        pw, fa = _cost(n, cg, cs, int(row_ptr[-1]), upper)
        assert pw >= 2 * fa


def test_plan_cuts_at_a_max_and_species_split_keys():
    # 3 groups of 50 keys, each sharing 10 with the previous group: 50 + 40 + 40 > 128 -> cut before group 2
    groups = [[(k + 1 + 40 * g, 29) for k in range(50)] for g in range(3)]
    rc, n, cg, cs, _, _, _ = _plan(groups, a_max=128)
    assert rc == 0 and list(cg) == [0, 2, 3] and list(cs) == [90, 50]
    rc, n, cg, cs, _, _, _ = _plan(groups, a_max=200)
    assert rc == 0 and list(cg) == [0, 3] and list(cs) == [130]
    # the same hash with another species code is another slot
    rc, n, cg, cs, rs, _, _ = _plan([[(5, 29), (5, 30), (5, 29)]])
    assert rc == 0 and list(cs) == [2] and list(rs) == [0, 1, 0]
    # a group alone above a_max: no plan
    rc, n, *_ = _plan([[(k, 29) for k in range(20)]], a_max=16)
    assert rc == 3 and n == 0
    # the group limit cuts as well
    rc, n, cg, *_ = _plan([[(1, 29)]] * 5, max_groups=2)
    assert rc == 0 and list(cg) == [0, 2, 4, 5]


def test_plan_collisions_get_their_own_slot():
    groups = [[(7, 29), (8, 29), (7, 29)], [(7, 29), (8, 29)]]
    rc, n, cg, cs, rs, rep, _ = _plan(groups)
    assert rc == 0 and n == 1 and list(cs) == [2] and list(rs) == [0, 1, 0, 0, 1]
    # rows 2 and 3 found different from their representative (row 0): each gets a slot of its own
    rc, n, cg, cs, rs, rep, _ = _plan(groups, unique=[0, 0, 1, 1, 0])
    assert rc == 0 and n == 1 and list(cs) == [4] and list(rs) == [0, 1, 2, 3, 1]
    assert list(rep) == [0, 1, 2, 3]


def test_no_sharing_keeps_the_pairwise_kernel():
    # one centre per structure (the add_structure regime): every group is a cluster of its own
    rng = np.random.default_rng(1)
    groups = [[(1000 * s + k + 1, 29) for k in range(int(rng.integers(20, 33)))] for s in range(200)]
    rc, n, cg, cs, _, _, row_ptr = _plan(groups)
    assert rc == 0 and n == 200
    for upper in (True, False):
        pw, fa = _cost(n, cg, cs, int(row_ptr[-1]), upper)
        assert pw < 2 * fa


@pytest.mark.parametrize("n_atoms, rows", [(32, 29), (108, 100)])
def test_cost_model_s5_s4_shapes(n_atoms, rows):
    # 340 x Cu32 (S5) and 200 x Cu108 (S4) shapes: the factored build executes several times fewer DMMAs
    n_struct = 340 if n_atoms == 32 else 200
    cg = np.arange(0, n_atoms * (n_struct + 1), n_atoms, dtype=np.int32)
    cs = np.full(n_struct, n_atoms, np.int32)
    pw, fa = _cost(n_struct, cg, cs, n_struct * n_atoms * rows, True)
    assert pw >= 5 * fa
