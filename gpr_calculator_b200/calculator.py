"""ASE calculator adapter (drop-in for gpr_calc/calculator.py:10-169, class GPR).

Host-side control only: it asks the GP surrogate (device hot path) for E, F and their standard
deviations, falls back to the base calculator when the uncertainty gate fails, queues the labelled
structure and refits on the reference's cadence.  The keyword arguments (``base, ff, save, tag, freq,
stress, f_tol, return_std``), the result keys, the printed "From Base model" / "From Surrogate" lines
and the abort on a bad refit are those of the reference.  With torch.distributed initialised, rank 0
runs the base calculator and broadcasts the labels (replaces the mpi4py bcast of calculator.py:58-59,90-91).
One keyword is added: ``stress_std=True`` (with ``stress=True``) also reports the standard deviation of the total
stress as ``results['var_s']`` (``get_var_s()``); the gate does not read it.

ASE is optional: with ASE installed ``GPR`` derives from ``ase.calculators.calculator.Calculator``;
without it a minimal stand-in base class provides the same ``parameters`` / ``results`` protocol so
that the adapter can be driven by any Atoms-like object (tests use utilities.SimpleAtoms).
"""
import sys

import numpy as np

from . import dist as gdist

try:   # pragma: no cover - depends on the environment
    from ase.calculators.calculator import Calculator, all_changes
    HAVE_ASE = True
except ImportError:
    HAVE_ASE = False
    all_changes = ['positions', 'numbers', 'cell', 'pbc', 'initial_charges', 'initial_magmoms']

    class _Parameters(dict):
        """dict with attribute access, like ase.calculators.calculator.Parameters"""

        def __getattr__(self, key):
            try:
                return self[key]
            except KeyError:
                raise AttributeError(key)

        def __setattr__(self, key, value):
            self[key] = value

    class Calculator:
        implemented_properties = []

        def __init__(self, **kwargs):
            self.parameters = _Parameters(kwargs)
            self.results = {}
            self.atoms = None

        def calculate(self, atoms=None, properties=('energy',), system_changes=all_changes):
            if atoms is not None:
                self.atoms = atoms.copy()

        def get_potential_energy(self, atoms=None):
            self.calculate(atoms)
            return self.results['energy']

        def get_forces(self, atoms=None):
            self.calculate(atoms)
            return self.results['forces']


def _fixed_indices(atoms):
    for c in getattr(atoms, "constraints", []) or []:
        if type(c).__name__ == "FixAtoms" and hasattr(c, "get_indices"):
            return c.get_indices()
    return []


def _bcast(obj):
    rank, size = gdist.world()
    if size == 1:
        return obj
    import torch.distributed as dist
    box = [obj]
    dist.broadcast_object_list(box, src=0)
    return box[0]


class GPR(Calculator):
    implemented_properties = ['energy', 'forces', 'stress', 'var_e', 'var_f', 'var_s']
    nolabel = True

    def __init__(self, **kwargs):
        Calculator.__init__(self, **kwargs)
        self.results = {}
        self.force_base = False
        self.allow_base = True
        self.update_gpr = True
        self.verbose = True
        self.ignore_E_std = True
        self.tag = self.parameters.tag if 'tag' in self.parameters else 'GPR'
        self.freq = self.parameters.freq if 'freq' in self.parameters else 10
        self.save = self.parameters.save if 'save' in self.parameters else True

    def freeze(self):
        self.allow_base = False
        self.update = False

    def unfreeze(self):
        self.update = True
        self.allow_base = True

    def calculate(self, atoms=None, properties=['energy', 'forces'], system_changes=all_changes):
        rank, _ = gdist.world()
        fix_ids = _fixed_indices(atoms)
        atoms.positions = _bcast(atoms.positions)
        gp_model = self.parameters.ff

        self._calculate(atoms, properties, system_changes)
        # uncertainty gate (calculator.py:62-73)
        e_tol = 100 if self.ignore_E_std else 1.2 * len(atoms) * gp_model.noise_e
        f_tol = 1.2 * gp_model.noise_f
        E_std, F_std = self.results['var_e'] * len(atoms), self.results['var_f'].max()
        E = self.results['energy']
        Fmax = np.abs(self.results['forces']).max()
        E_fail = E_std > e_tol
        f_ref = max(f_tol, Fmax / 2.5)
        force_fail = not (F_std < f_ref).all()

        if self.force_base or (self.allow_base and (E_fail or force_fail)):
            gp_model.use_base += 1
            if rank == 0:
                atoms.calc = self.parameters.base
                eng = atoms.get_potential_energy()
                forces = atoms.get_forces()
                forces[fix_ids] = 0.0
                atoms.calc = None
                data = (atoms.copy(), eng, forces)
                f_max = np.abs(forces).max()
                print(f"From Base model E: {E_std:.3f}/{E:.3f}/{eng:.3f}, F: {F_std:.3f}/{Fmax:.3f}/{f_max:.3f}")
            else:
                data, eng, forces = None, None, None
            data, eng, forces = _bcast((data, eng, forces))
            gp_model.add_structure(data)
            self.results["energy"] = eng
            self.results["forces"] = forces
            atoms.calc = self
        else:
            gp_model.use_surrogate += 1
            if rank == 0:
                print(f"From Surrogate  E: {E_std:.3f}/{e_tol:.3f}/{E:.3f}, F: {F_std:.3f}/{f_tol:.3f}/{Fmax:.3f}")

        # refit cadence (calculator.py:101-117)
        freq = max([2, self.freq // 2]) if gp_model.N_forces > 100 else self.freq
        if self.update_gpr and (gp_model.N_queue > freq or gp_model.N_energy_queue >= 2):
            gp_model.fit(opt=True, show=False, maxiter=10)
            if rank == 0 and self.save:
                gp_model.save(f'{self.tag}-gpr.json', f'{self.tag}-gpr.db', verbose=False)
                print(gp_model)
            gp_model.validate_data(show=True)
            if gp_model.error['energy_mae'] > 0.1 or gp_model.error['forces_mae'] > 0.3:
                print("ERROR: The error is too large, check the data.")
                print(gp_model.error)
                print("The program stops here!\n")
                sys.exit()

    def _calculate(self, atoms, properties, system_changes):
        """E / F (/ std) from the GPR model (calculator.py:119-155)."""
        Calculator.calculate(self, atoms, properties, system_changes)
        stress = self.parameters.stress if 'stress' in self.parameters else False
        f_tol = self.parameters.f_tol if 'f_tol' in self.parameters else 1e-12
        return_std = self.parameters.return_std if 'return_std' in self.parameters else True
        stress_std = self.parameters.stress_std if 'stress_std' in self.parameters else False
        if stress and stress_std:
            # total stress and its standard deviation from one row per atom (GP.predict_structures(stress=True))
            res = self.parameters.ff.predict_structures([atoms], return_std=True, f_tol=f_tol, stress=True)[0]
            self.results['var_e'] = res[3]
            self.results['var_f'] = res[4]
            self.results['var_s'] = res[5]
            self.results['stress'] = res[2]
        else:
            res = self.parameters.ff.predict_structure(atoms, stress, return_std, f_tol=f_tol)
            if return_std:
                self.results['var_e'] = res[3]
                self.results['var_f'] = res[4]
            self.results['stress'] = res[2].sum(axis=0) if stress else None
        self.results['energy'] = res[0]
        self.results['free_energy'] = res[0]
        self.results['forces'] = res[1]
        self.forces = res[1]

    def get_var_e(self, total=False):
        if total:
            return self.results["var_e"] * len(self.results["forces"])   # eV
        return self.results["var_e"]                                       # eV/atom

    def get_var_f(self):
        return self.results["var_f"]

    def get_var_s(self):
        """Standard deviation [6] of the total stress (xx, yy, zz, xy, xz, yz); set when GPR(stress=True, stress_std=True)."""
        return self.results["var_s"]

    def get_e(self, peratom=True):
        if peratom:
            return self.results["energy"] / len(self.results["forces"])
        return self.results["energy"]
