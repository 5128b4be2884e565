"""RBF many-body kernel object (drop-in for gpr_calc/kernels/RBF_mb.py:7-524) on the B200.

    k(x_i, x_j) = sigma^2 exp(-(1 - (x^_i . x^_j)^zeta) / (2 l^2))

Same constructor, attributes and methods as the reference class.  The blocks K_ee / K_ef / K_ff,
their dK/dl and the diagonal are computed by libgpr_b200.so and assembled on device; the public
methods return numpy arrays, the ``*_device`` methods return torch CUDA tensors (what GP.fit /
GP.predict use so that K never leaves HBM).  The reference's mpi4py row split
(RBF_mb.py:257-301, 348-431, 471-521) is replaced by the ``window`` argument (row-block sharding).
"""
import numpy as np

from .. import _lib
from ..device import packs_of, k_total_device, k_total_stress_device, diag_device, k_virial_device, virial_packs


class RBF_mb():
    def __init__(self,
                 para=[1., 1.],
                 bounds=[[1e-2, 5e+1], [1e-1, 1e+1]],
                 zeta=2,
                 ncpu=1,
                 device='cuda'):
        self.name = 'RBF'
        self.bounds = bounds
        self.update(para)
        self.zeta = zeta
        self.device = device
        self.ncpu = ncpu

    def __str__(self):
        return "{:.5f}**2 *RBF({:.5f})".format(self.sigma, self.l)

    def load_from_dict(self, dict0):
        self.sigma = dict0["sigma"]
        self.l = dict0["l"]
        self.zeta = dict0["zeta"]
        self.bounds = dict0["bounds"]
        self.name = dict0["name"]

    def save_dict(self):
        return {"name": self.name, "sigma": self.sigma, "l": self.l, "zeta": self.zeta, "bounds": self.bounds}

    def parameters(self):
        return [self.sigma, self.l]

    def update(self, para):
        self.sigma, self.l = para[0], para[1]

    # ---- device entry points ------------------------------------------------------------------
    def cov_args(self, grad=False, f_tol=1e-10):
        """Arguments of device.build_energy_rows / build_force_rows for this kernel (row-sharded builds)."""
        return dict(kernel=_lib.RBF, p0=float(self.sigma), p1=float(self.l), zeta=float(self.zeta), zeta_ef=float(self.zeta),
                    zeta_ff=float(self.zeta), use_tol=not grad, tol=f_tol, has_dk=True)

    def k_total_device(self, data1, data2=None, f_tol=1e-10, grad=False, window=None, symmetric=True):
        """(K, dK/dl) as CUDA tensors.  grad=True follows k_total_with_grad: no pair cut in K_ff
        (rbf_kernel.cpp:534); grad=False follows k_total: pair cut `dK_dD > f_tol` (:395)."""
        side1 = packs_of(data1)
        side2 = None if data2 is None else packs_of(data2)
        return k_total_device(_lib.RBF, float(self.sigma), float(self.l), float(self.zeta), side1, side2,
                              use_tol=not grad, tol=f_tol, grad=grad, window=window, symmetric=symmetric)

    def diag_device(self, data, _packed_ok=True):
        """Energy rows: eps-regularised formula of kernels/base.py:107-130; force rows: diagonal of
        the (I, I) block with kff_C's default tol = 1e-12 (RBF_mb.py:103-110)."""
        return diag_device(_lib.RBF, float(self.sigma), float(self.l), float(self.zeta), packs_of(data), tol=1e-12)

    # ---- reference API (numpy in / numpy out) --------------------------------------------------
    def diag(self, data):
        """Diagonal of k(X, X) (RBF_mb.py:62-133)."""
        return self.diag_device(data).cpu().numpy()

    def k_total(self, data1, data2=None, f_tol=1e-10):
        """Covariance between data1 and data2 (training K when data2 is None) (RBF_mb.py:135-171)."""
        K, _ = self.k_total_device(data1, data2, f_tol=f_tol, grad=False)
        return K.cpu().numpy()

    def k_total_with_grad(self, data1, f_tol=1e-10):
        """K and dK/d(sigma, l) stacked on the last axis (RBF_mb.py:173-204)."""
        K, dK_l = self.k_total_device(data1, None, f_tol=f_tol, grad=True)
        K = K.cpu().numpy()
        return K, np.dstack(((2 / self.sigma) * K, dK_l.cpu().numpy()))

    def k_total_stress_device(self, data1, data2, tol=1e-10):
        """(K, K1) as CUDA tensors; K1 holds the 6 Voigt stress rows of every force item of data1."""
        return k_total_stress_device(_lib.RBF, float(self.sigma), float(self.l), float(self.zeta), data1, data2,
                                     use_tol=True, tol=tol)

    def k_virial_device(self, V, data2, tol=1e-10):
        """(K*, prior variance) of the total stress rows of the stress tuple V (batch.virial_rows_from_batch): K* with the
        pair cut of k_total_stress_device, the prior with the force-row tol of diag_device."""
        return k_virial_device(_lib.RBF, float(self.sigma), float(self.l), float(self.zeta), virial_packs(V), packs_of(data2),
                               use_tol=True, tol=tol, prior_tol=1e-12)

    def k_total_with_stress(self, data1, data2, tol=1e-10):
        """Covariance for energy / force / stress prediction (RBF_mb.py:206-229): data1's force items carry
        9 columns (3 force + 6 Voigt).  Returns (C, C1) with C1 = [C_se, C_sf]."""
        K, K1 = self.k_total_stress_device(data1, data2, tol=tol)
        return K.cpu().numpy(), (None if K1 is None else K1.cpu().numpy())
