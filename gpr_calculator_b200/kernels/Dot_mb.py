"""Dot (polynomial) many-body kernel object (drop-in for gpr_calc/kernels/Dot_mb.py:5-173).

    k(x_i, x_j) = sigma^2 ((x^_i . x^_j)^zeta + sigma0^2)

Reference quirks reproduced on purpose (SURVEY.md §7.3):
  * k_total passes zeta in the sigma0 slot of kef_C / kff_C, so the E-F and F-F blocks use
    zeta = 2 while the E-E block uses self.zeta (Dot_mb.py:108-117 vs dot_kernel.py:66,162);
    k_total_with_grad uses self.zeta everywhere (Dot_mb.py:138-143);
  * d/dsigma0 is the constant 0.8 * 2 sigma^2 sigma0 on the E-E block and 0 elsewhere
    (dot_kernel.py:58,154,265);
  * diag() accepts force data only as a list / object array of (x, dxdr, ele) (Dot_mb.py:71-78).
"""
import numpy as np
import torch

from .. import _lib
from ..device import (packs_of, k_total_device, k_total_stress_device, diag_device, energy_pack, force_pack,
                      k_virial_device, virial_packs)


class Dot_mb():
    def __init__(self, para=[1., 1.], bounds=[[1e-2, 5e+1], [1e-2, 1e+1]], zeta=3, device="cuda"):
        self.name = 'Dot'
        self.bounds = bounds
        self.update(para)
        self.zeta = zeta
        self.device = device

    def __str__(self):
        return "{:.3f}**2 *Dot({:.3f})".format(self.sigma, self.sigma0)

    def load_from_dict(self, dict0):
        self.sigma = dict0["sigma"]
        self.sigma0 = dict0["sigma0"]
        self.zeta = dict0["zeta"]
        self.bounds = dict0["bounds"]
        self.name = dict0["name"]

    def save_dict(self):
        return {"name": self.name, "sigma": self.sigma, "sigma0": self.sigma0, "zeta": self.zeta,
                "bounds": self.bounds}

    def parameters(self):
        return [self.sigma, self.sigma0]

    def update(self, para):
        self.sigma, self.sigma0 = para[0], para[1]

    # ---- device entry points ------------------------------------------------------------------
    def cov_args(self, grad=False, f_tol=1e-12):
        """Arguments of device.build_energy_rows / build_force_rows (see the module docstring for the
        zeta used by the E-F / F-F blocks)."""
        z_cross = float(self.zeta) if grad else 2.0
        return dict(kernel=_lib.DOT, p0=float(self.sigma), p1=float(self.sigma0), zeta=float(self.zeta), zeta_ef=z_cross,
                    zeta_ff=z_cross, use_tol=False, tol=0.0, has_dk=False)

    def k_total_device(self, data1, data2=None, f_tol=1e-12, grad=False, window=None, symmetric=True):
        """(K, None).  grad selects which zeta the E-F / F-F blocks use (see module docstring);
        the gradient blocks themselves are closed-form (grad_terms)."""
        side1 = packs_of(data1)
        side2 = None if data2 is None else packs_of(data2)
        z_cross = float(self.zeta) if grad else 2.0
        K, _ = k_total_device(_lib.DOT, float(self.sigma), float(self.sigma0), float(self.zeta), side1, side2,
                              use_tol=False, tol=0.0, grad=False, zeta_ef=z_cross, zeta_ff=z_cross,
                              window=window, symmetric=symmetric)
        return K, None

    def diag_device(self, data, _packed_ok=False):
        if "force" in data and isinstance(data["force"], tuple) and not _packed_ok:
            raise ValueError("Dot_mb.diag expects force data as a list of (x, dxdr, ele) (Dot_mb.py:71-78)")
        # the numpy K_ff behind Dot_mb.diag regularises every norm with +1e-8 (Dot_mb.py:206-221)
        e = energy_pack(data["energy"]) if "energy" in data else None
        f = force_pack(data["force"], norm_eps=1e-8) if "force" in data else None
        return diag_device(_lib.DOT, float(self.sigma), float(self.sigma0), float(self.zeta), (e, f), tol=0.0)

    # ---- reference API ------------------------------------------------------------------------
    def diag(self, data):
        return self.diag_device(data).cpu().numpy()

    def k_total(self, data1, data2=None, tol=1e-12):
        K, _ = self.k_total_device(data1, data2, grad=False)
        return K.cpu().numpy()

    def k_total_with_grad(self, data1):
        K, _ = self.k_total_device(data1, None, grad=True)
        K = K.cpu().numpy()
        NE = len(data1["energy"][-1]) if isinstance(data1.get("energy"), tuple) else len(data1.get("energy", []))
        C2 = np.zeros(K.shape)
        C2[:NE, :NE] = 0.8 * 2 * self.sigma ** 2 * self.sigma0
        return K, np.dstack((2 * K / self.sigma, C2))

    def k_total_stress_device(self, data1, data2, tol=1e-10):
        # same zeta-in-the-sigma0-slot quirk as k_total: the cross blocks use zeta = 2 (Dot_mb.py:166-170)
        return k_total_stress_device(_lib.DOT, float(self.sigma), float(self.sigma0), float(self.zeta), data1, data2,
                                     use_tol=False, tol=0.0, zeta_ef=2.0, zeta_ff=2.0)

    def k_virial_device(self, V, data2, tol=1e-10):
        """(K*, prior variance) of the total stress rows of V: K* with k_total_stress_device's cross-block zeta = 2, the
        prior as diag_device builds force rows (norm_eps = 1e-8, self.zeta)."""
        return k_virial_device(_lib.DOT, float(self.sigma), float(self.sigma0), float(self.zeta), virial_packs(V),
                               packs_of(data2), use_tol=False, tol=0.0, zeta_ef=2.0, zeta_ff=2.0,
                               prior_packs=virial_packs(V, norm_eps=1e-8), prior_tol=0.0)

    def k_total_with_stress(self, data1, data2, tol=1e-10):
        """Dot_mb.py:150-173 (tol is not used there either)."""
        K, K1 = self.k_total_stress_device(data1, data2)
        return K.cpu().numpy(), (None if K1 is None else K1.cpu().numpy())
