"""CPU ORACLE (test infrastructure only) — numpy/scipy restatement of the kernel objects and the
GP algebra of the reference (gpr_calc/kernels/RBF_mb.py, Dot_mb.py, kernels/base.py,
gaussianprocess.py:128-202, 286-317, 319-379, 834-918) on top of oracle/kernels.py.

Parity status: PINNED by tests/golden/{kernels,gp}.npz, produced by the reference itself
(tests/golden/gen_golden.py).  Only tests/, smoke() and bench.py's cpu_baseline leg import this.
"""
import numpy as np
from scipy.linalg import cholesky, cho_solve, solve_triangular

from .kernels import RBFOracle, DotOracle, list_to_tuple


def build_covariance(c_ee, c_ef, c_fe, c_ff):
    """kernels/base.py:3-30"""
    have = [x is not None for x in (c_ee, c_ef, c_fe, c_ff)]
    if all(have):
        return np.block([[c_ee, c_ef], [c_fe, c_ff]])
    if have == [False, False, True, True]:
        return np.hstack((c_fe, c_ff))
    if have == [True, True, False, False]:
        return np.hstack((c_ee, c_ef))
    for x in (c_ef, c_ee, c_ff, c_fe):
        if x is not None and sum(have) == 1:
            return x
    return None


def _present(data, key):
    if key not in data:
        return False
    v = data[key]
    return len(v[-1]) > 0 if isinstance(v, tuple) else len(v) > 0


class RBFKernelOracle:
    """RBF_mb.k_total / k_total_with_grad / diag (RBF_mb.py:62-204), single rank."""

    def __init__(self, para=(1.0, 1.0), zeta=2, backend="port"):
        self.sigma, self.l = para
        self.zeta = zeta
        self.k = RBFOracle(backend)

    def update(self, para):
        self.sigma, self.l = para[0], para[1]

    def parameters(self):
        return [self.sigma, self.l]

    def k_total(self, data1, data2=None, f_tol=1e-10):
        same = data2 is None
        if same:
            data2 = data1
        s, l, z = self.sigma, self.l, self.zeta
        C_ee = C_ef = C_fe = C_ff = None
        if _present(data1, "energy") and _present(data2, "energy"):
            C_ee = self.k.kee_C(data1["energy"], data2["energy"], s, l, z)
        if _present(data1, "energy") and _present(data2, "force"):
            C_ef = self.k.kef_C(data1["energy"], data2["force"], s, l, z)
        if _present(data1, "force") and _present(data2, "energy"):
            C_fe = C_ef.T if same else self.k.kef_C(data2["energy"], data1["force"], s, l, z, transpose=True)
        if _present(data1, "force") and _present(data2, "force"):
            C_ff = self.k.kff_C(data1["force"], data2["force"], s, l, z, tol=f_tol)
        return build_covariance(C_ee, C_ef, C_fe, C_ff)

    def k_total_with_grad(self, data1):
        s, l, z = self.sigma, self.l, self.zeta
        ee = self.k.kee_C(data1["energy"], data1["energy"], s, l, z, grad=True)
        ef = self.k.kef_C(data1["energy"], data1["force"], s, l, z, grad=True)
        ff = self.k.kff_C(data1["force"], data1["force"], s, l, z, grad=True)
        mats = [build_covariance(ee[i], ef[i], ef[i].T, ff[i]) for i in range(3)]
        return mats[0], np.dstack((mats[1], mats[2]))

    def diag(self, data):
        """Energy rows: kernels/base.py:107-130 (eps-regularised); force rows: diagonal of
        kff_C(dat, dat) with the default tol = 1e-12 (RBF_mb.py:103-110)."""
        s2, l2, z = self.sigma ** 2, self.l ** 2, self.zeta
        parts = []
        if "energy" in data:
            e = data["energy"]
            if isinstance(e, list):
                e = list_to_tuple(e, mode="energy")
            X, ELE, ind = e
            out, c = np.zeros(len(ind)), 0
            for i, n in enumerate(ind):
                x, ele = X[c:c + n], np.asarray(ELE[c:c + n])
                nrm = np.linalg.norm(x, axis=1) + 1e-8
                dd = (x @ x.T) / (1e-8 + nrm[:, None] * nrm[None, :])
                k = s2 * np.exp(-(0.5 / l2) * (1 - dd ** z))
                k[ele[:, None] != ele[None, :]] = 0
                out[i] = k.sum() / (n * n)
                c += n
            parts.append(out)
        if "force" in data:
            f = data["force"]
            if isinstance(f, (list, np.ndarray)):
                f = list_to_tuple(list(f))
            X, dX, ELE, ind = f
            out, c = np.zeros(3 * len(ind)), 0
            for i, n in enumerate(ind):
                dat = (X[c:c + n], dX[c:c + n], ELE[c:c + n], [n])
                out[3 * i:3 * i + 3] = np.diag(self.k.kff_C(dat, dat, self.sigma, self.l, self.zeta))
                c += n
            parts.append(out)
        return np.hstack(parts)


class DotKernelOracle:
    """Dot_mb.k_total / k_total_with_grad (Dot_mb.py:87-148) including the zeta-slot quirk."""

    def __init__(self, para=(1.0, 1.0), zeta=3, backend="port"):
        self.sigma, self.sigma0 = para
        self.zeta = zeta
        self.k = DotOracle(backend)

    def update(self, para):
        self.sigma, self.sigma0 = para[0], para[1]

    def parameters(self):
        return [self.sigma, self.sigma0]

    def k_total(self, data1, data2=None):
        same = data2 is None
        if same:
            data2 = data1
        s, s0, z = self.sigma, self.sigma0, self.zeta
        C_ee = C_ef = C_fe = C_ff = None
        if _present(data1, "energy") and _present(data2, "energy"):
            C_ee = self.k.kee_C(data1["energy"], data2["energy"], s, s0, z)
        if _present(data1, "energy") and _present(data2, "force"):
            C_ef = self.k.kef_C(data1["energy"], data2["force"], s, z)          # zeta lands in sigma0: zeta = 2
        if _present(data1, "force") and _present(data2, "energy"):
            C_fe = C_ef.T if same else self.k.kef_C(data2["energy"], data1["force"], s, z, transpose=True)
        if _present(data1, "force") and _present(data2, "force"):
            C_ff = self.k.kff_C(data1["force"], data2["force"], s, z)
        return build_covariance(C_ee, C_ef, C_fe, C_ff)

    def k_total_with_grad(self, data1):
        s, s0, z = self.sigma, self.sigma0, self.zeta
        ee = self.k.kee_C(data1["energy"], data1["energy"], s, s0, z, grad=True)
        ef = self.k.kef_C(data1["energy"], data1["force"], s, s0, z, grad=True)
        ff = self.k.kff_C(data1["force"], data1["force"], s, s0, z, grad=True)
        mats = [build_covariance(ee[i], ef[i], ef[i].T, ff[i]) for i in range(3)]
        return mats[0], np.dstack((mats[1], mats[2]))


def add_noise(K, NE, noise_e, noise_f):
    K = K.copy()
    idx = np.arange(len(K))
    K[idx[:NE], idx[:NE]] += noise_e ** 2
    K[idx[NE:], idx[NE:]] += noise_f ** 2
    return K


def lml_from_matrices(K, dK, y_train, NE, noise_e, noise_f):
    """The algebra of gaussianprocess.py:162-198 on given matrices: K is the noise-free covariance [N, N] (the first NE
    rows are energy rows), dK[:, :, k] = dK/dtheta_k (None: no gradient), y_train [N] or [N, 1].
    Returns the LML, or (LML, gradient) when dK is given."""
    y_train = np.asarray(y_train, dtype=np.float64).reshape(len(K), -1)
    K = add_noise(K, NE, noise_e, noise_f)
    L = cholesky(K, lower=True)
    alpha = cho_solve((L, True), y_train)
    mll = -0.5 * float(y_train[:, 0] @ alpha[:, 0]) - np.log(np.diag(L)).sum() - len(K) / 2 * np.log(2 * np.pi)
    if dK is None:
        return mll
    W = alpha @ alpha.T - cho_solve((L, True), np.eye(len(K)))
    grad = 0.5 * np.einsum("ij,jik->k", W, dK)
    return mll, grad


def log_marginal_likelihood(kernel, train_x, y_train, noise_e, noise_f, eval_gradient=True):
    """gaussianprocess.py:160-202 with fixed noise (noise_bounds is None)."""
    NE = len(train_x["energy"][-1]) if len(train_x["energy"]) > 0 else 0
    if eval_gradient:
        K, dK = kernel.k_total_with_grad(train_x)
    else:
        K, dK = kernel.k_total(train_x), None
    return lml_from_matrices(K, dK, y_train, NE, noise_e, noise_f)


def fit_factors(kernel, train_x, y_train, noise_e, noise_f):
    """gaussianprocess.py:286-299, 128-131: K (pair-cut variant), L, alpha, explicit K^-1."""
    NE = len(train_x["energy"][-1]) if len(train_x["energy"]) > 0 else 0
    K = add_noise(kernel.k_total(train_x), NE, noise_e, noise_f)
    L = cholesky(K, lower=True)
    alpha = cho_solve((L, True), y_train)
    L_inv = solve_triangular(L.T, np.eye(len(L)))
    return L, alpha, L_inv @ L_inv.T


def predict_rows(kernel, X, train_x, alpha, K_inv, f_tol=1e-10, return_std=False):
    """gaussianprocess.py:335-377 / 878-908: mean and clipped std of the rows of X."""
    K_trans = kernel.k_total(X, train_x, f_tol) if isinstance(kernel, RBFKernelOracle) else kernel.k_total(X, train_x)
    mean = (K_trans @ alpha)[:, 0]
    if not return_std:
        return mean
    var = kernel.diag(X) - np.einsum("ij,ij->i", K_trans @ K_inv, K_trans)
    var[var < 0] = 0.0
    return mean, np.sqrt(var)
