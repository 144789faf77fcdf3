"""Calculator shim and minimal host-side MD / relaxation drivers (SURVEY.md §8 row f2, host stage).

``CHGNetCalculator`` mirrors the reference's ASE calculator (chgnet/model/dynamics.py:58-181): same
constructor keywords, ``calculate(atoms, properties, system_changes, task)``, the same ``results`` keys
and unit conventions (total energy in eV, forces in eV/A, stress x ``stress_weight`` = eV/A^3 as a 3x3
array, ``magmoms``, ``free_energy``, ``crystal_fea``, optional ``energies``).  When ``ase`` is installed
it subclasses ``ase.calculators.calculator.Calculator`` and can be attached to ``ase.Atoms``; without
``ase`` it is a plain object that accepts anything with ``get_atomic_numbers() / get_positions() /
get_cell()`` (e.g. :class:`Atoms` below), so ``VelocityVerlet`` and ``fire_relax`` here run stand-alone.

Every step rebuilds the graph with the native host builder (``chg_graph_build``) and runs one
``chg_forward``; keeping positions / velocities on the device and building the graph there is the next
stage of this row.
"""
from __future__ import annotations

import numpy as np

from chgnet_b200 import PredTask

GPA = 1.0 / 160.21766208  # GPa -> eV/A^3 (ase.units.GPa)
FS = 0.09822694788464063  # fs in ASE time units (A sqrt(amu/eV))  (ase.units.fs)
KB = 8.617333262e-5  # eV/K

# standard atomic weights, Z = 1..94 (amu)
ATOMIC_MASSES = np.array([
    1.008, 4.002602, 6.94, 9.0121831, 10.81, 12.011, 14.007, 15.999, 18.998403163, 20.1797, 22.98976928, 24.305, 26.9815385,
    28.085, 30.973761998, 32.06, 35.45, 39.948, 39.0983, 40.078, 44.955908, 47.867, 50.9415, 51.9961, 54.938044, 55.845,
    58.933194, 58.6934, 63.546, 65.38, 69.723, 72.630, 74.921595, 78.971, 79.904, 83.798, 85.4678, 87.62, 88.90584, 91.224,
    92.90637, 95.95, 97.90721, 101.07, 102.90550, 106.42, 107.8682, 112.414, 114.818, 118.710, 121.760, 127.60, 126.90447,
    131.293, 132.90545196, 137.327, 138.90547, 140.116, 140.90766, 144.242, 144.91276, 150.36, 151.964, 157.25, 158.92535,
    162.500, 164.93033, 167.259, 168.93422, 173.054, 174.9668, 178.49, 180.94788, 183.84, 186.207, 190.23, 192.217, 195.084,
    196.966569, 200.592, 204.38, 207.2, 208.98040, 208.98243, 209.98715, 222.01758, 223.01974, 226.02541, 227.02775, 232.0377,
    231.03588, 238.02891, 237.04817, 244.06421])

try:  # optional: real ASE base class
    from ase.calculators.calculator import Calculator as _Base
    from ase.calculators.calculator import all_changes, all_properties
except ImportError:  # stand-alone
    all_changes, all_properties = ["positions", "numbers", "cell", "pbc"], ["energy", "forces", "stress", "magmoms"]

    class _Base:  # the two things the shim needs from ase's Calculator
        def __init__(self, **_: object) -> None:
            self.results: dict = {}
            self.atoms = None

        def calculate(self, atoms=None, properties=None, system_changes=None) -> None:
            if atoms is not None:
                self.atoms = atoms


class Atoms:
    """Minimal periodic structure (numbers, Cartesian positions in A, cell rows = lattice vectors)."""

    def __init__(self, numbers, positions, cell, velocities=None) -> None:
        self.numbers = np.asarray(numbers, dtype=np.int64)
        self.positions = np.asarray(positions, dtype=np.float64).reshape(-1, 3)
        self.cell = np.asarray(cell, dtype=np.float64).reshape(3, 3)
        self.velocities = np.zeros_like(self.positions) if velocities is None else np.asarray(velocities, dtype=np.float64)
        self.calc = None

    def get_atomic_numbers(self):
        return self.numbers

    def get_positions(self):
        return self.positions

    def get_cell(self):
        return self.cell

    def get_masses(self):
        return ATOMIC_MASSES[self.numbers - 1]

    def get_volume(self) -> float:
        return abs(float(np.linalg.det(self.cell)))

    def set_cell(self, cell, scale_atoms: bool = False) -> None:
        """New cell; ``scale_atoms=True`` keeps the fractional coordinates (ase's ``Atoms.set_cell``)."""
        cell = np.asarray(cell, dtype=np.float64).reshape(3, 3)
        if scale_atoms:
            self.positions = (self.positions @ np.linalg.inv(self.cell)) @ cell
        self.cell = cell.copy()

    def __len__(self) -> int:
        return len(self.numbers)


class CHGNetCalculator(_Base):
    """CHGNet calculator (reference dynamics.py:58-181) on the B200 kernel path."""

    implemented_properties = ("energy", "forces", "stress", "magmoms", "energies")

    def __init__(self, model=None, *, use_device: str | None = None, check_cuda_mem: bool = False,
                 stress_weight: float = GPA, on_isolated_atoms: str = "warn", return_site_energies: bool = False,
                 **kwargs) -> None:
        super().__init__(**kwargs)
        from chgnet_b200.model import CHGNet

        self.model = model if model is not None else CHGNet.load(use_device=use_device, verbose=False)
        if use_device is not None:
            self.model = self.model.to(use_device)
        self.device = self.model.device
        self.stress_weight = stress_weight
        self.return_site_energies = return_site_energies
        self.on_isolated_atoms = on_isolated_atoms
        del check_cuda_mem

    @classmethod
    def from_file(cls, path: str, use_device: str | None = None, **kwargs):
        from chgnet_b200.model import CHGNet

        return cls(model=CHGNet.from_file(path), use_device=use_device, **kwargs)

    @property
    def version(self) -> str | None:
        return self.model.version

    @property
    def n_params(self) -> int:
        return self.model.n_params

    def calculate(self, atoms=None, properties=None, system_changes=None, task: PredTask = "efsm") -> None:
        properties = properties or all_properties
        system_changes = system_changes or all_changes
        super().calculate(atoms=atoms, properties=properties, system_changes=system_changes)
        atoms = atoms if atoms is not None else self.atoms
        numbers = np.asarray(atoms.get_atomic_numbers())
        cell = np.asarray(atoms.get_cell(), dtype=np.float64).reshape(3, 3)
        frac = np.asarray(atoms.get_positions(), dtype=np.float64) @ np.linalg.inv(cell)
        from chgnet_b200 import graphgen

        graph = graphgen.make_crystal_graph(numbers, frac, cell, atom_graph_cutoff=self.model.graph_converter.atom_graph_cutoff,
                                            bond_graph_cutoff=self.model.graph_converter.bond_graph_cutoff)
        if self.on_isolated_atoms != "ignore":
            centers = graph.atom_graph[:, 0].tolist() if graph.atom_graph.dim() == 2 else []
            isolated = set(range(len(numbers))) - set(centers)
            if isolated:
                msg = f"structure has isolated atoms {sorted(isolated)} (no neighbour within the atom-graph cutoff)"
                if self.on_isolated_atoms == "error":
                    raise ValueError(msg)
                import warnings

                warnings.warn(msg, stacklevel=2)
        pred = self.model.predict_graph(graph, task=task, return_crystal_feas=True,
                                        return_site_energies=self.return_site_energies)
        extensive = len(numbers) if self.model.is_intensive else 1
        key_map = {"e": ("energy", extensive), "f": ("forces", 1), "m": ("magmoms", 1), "s": ("stress", self.stress_weight)}
        self.results = {**getattr(self, "results", {}),
                        **{long: pred[k] * fac for k, (long, fac) in key_map.items() if k in pred}}
        self.results["free_energy"] = self.results["energy"]
        self.results["crystal_fea"] = pred["crystal_fea"]
        if self.return_site_energies:
            self.results["energies"] = pred["site_energies"]


class VelocityVerlet:
    """NVE molecular dynamics on the host (the integrator of ase.md.verlet restated): one calculator
    call per step.  ``timestep`` in fs."""

    def __init__(self, atoms, calculator: CHGNetCalculator, timestep: float = 2.0, task: PredTask = "ef") -> None:
        self.atoms, self.calc, self.dt, self.task = atoms, calculator, timestep * FS, task
        self.calc.calculate(atoms, task=task)
        self.forces = np.asarray(self.calc.results["forces"], dtype=np.float64)
        self.nsteps = 0

    def kinetic_energy(self) -> float:
        return float(0.5 * (self.atoms.get_masses()[:, None] * self.atoms.velocities**2).sum())

    def potential_energy(self) -> float:
        return float(self.calc.results["energy"])

    def temperature(self) -> float:
        return 2.0 * self.kinetic_energy() / (3.0 * len(self.atoms) * KB)

    def set_temperature(self, kelvin: float, seed: int = 0) -> None:
        rng = np.random.default_rng(seed)
        m = self.atoms.get_masses()[:, None]
        v = rng.normal(size=self.atoms.positions.shape) * np.sqrt(KB * kelvin / m)
        v -= (m * v).sum(axis=0) / m.sum()  # no centre-of-mass drift
        self.atoms.velocities = v

    def run(self, steps: int) -> list[dict]:
        log = []
        m = self.atoms.get_masses()[:, None]
        for _ in range(steps):
            self.atoms.velocities = self.atoms.velocities + 0.5 * self.dt * self.forces / m
            self.atoms.positions = self.atoms.positions + self.dt * self.atoms.velocities
            self.calc.calculate(self.atoms, task=self.task)
            self.forces = np.asarray(self.calc.results["forces"], dtype=np.float64)
            self.atoms.velocities = self.atoms.velocities + 0.5 * self.dt * self.forces / m
            self.nsteps += 1
            log.append({"step": self.nsteps, "e_pot": self.potential_energy(), "e_kin": self.kinetic_energy(),
                        "temperature": self.temperature()})
        return log


def berendsen_lambda(temperature: float, target: float, dt_over_taut: float) -> float:
    """Velocity scale of ASE's ``NVTBerendsen.scale_velocities``: sqrt(1 + (T0 / T - 1) dt / tau_t) clamped to
    [0.9, 1.1]; 1.1 at T = 0 (ASE divides by zero there and clamps the infinity)."""
    if temperature == 0.0:
        return 1.1
    a = 1.0 + (target / temperature - 1.0) * dt_over_taut
    return 0.9 if a <= 0.81 else min(max(float(np.sqrt(a)), 0.9), 1.1)


class NVTBerendsen(VelocityVerlet):
    """Berendsen NVT on the host (ASE's ``NVTBerendsen``, the reference's default ensemble, dynamics.py:595-609),
    the checker of ``DeviceMD(ensemble="nvt")``.  One step, with F (and the stress) of the previous call:

    1. thermostat: T = K_tr / (3 N k_B), v <- lambda v (``berendsen_lambda``);
    2. barostat (the NPT subclasses): P_a = -sigma_aa + K_aa / V, then the cell is scaled with the atoms;
    3. v <- v + dt/2 F/m;  4. ``fix_com``: v_i <- v_i - mean(m v) / m_i;  5. x <- x + dt v;
    6. one ``calculate`` (forces, stress);  7. v <- v + dt/2 F/m.

    ``temperature`` in K, ``pressure`` / ``bulk_modulus`` in GPa, ``timestep`` / ``taut`` / ``taup`` in fs.  Any object
    with ``calculate(atoms, task=...)`` and ``results`` {"energy", "forces", "stress" (eV/A^3)} can drive it."""

    barostat: str | None = None

    def __init__(self, atoms, calculator, timestep: float = 2.0, temperature: float = 300.0, taut: float | None = None,
                 fix_com: bool = True, task: PredTask | None = None) -> None:
        self.fix_com = fix_com
        self.target_temperature = float(temperature)
        self.dt_over_taut = (timestep * FS) / ((100.0 * timestep if taut is None else taut) * FS)
        super().__init__(atoms, calculator, timestep=timestep, task=task or ("efs" if self.barostat else "ef"))
        self.stress = self._stress()

    def _stress(self) -> np.ndarray | None:
        if self.barostat is None:
            return None
        return np.asarray(self.calc.results["stress"], dtype=np.float64).reshape(3, 3)

    def set_target(self, temperature: float | None = None, pressure: float | None = None) -> None:
        if temperature is not None:
            self.target_temperature = float(temperature)
        if pressure is not None:
            self.target_pressure = float(pressure) * GPA

    def scale_cell(self) -> None:
        """The barostat (NPT subclasses)."""

    def step(self) -> None:
        atoms, m = self.atoms, self.atoms.get_masses()[:, None]
        self.last_lambda = berendsen_lambda(self.temperature(), self.target_temperature, self.dt_over_taut)
        atoms.velocities = self.last_lambda * atoms.velocities
        self.scale_cell()
        v = atoms.velocities + 0.5 * self.dt * self.forces / m
        if self.fix_com:
            p = m * v
            v = (p - p.sum(axis=0) / len(p)) / m
        atoms.velocities = v
        atoms.positions = atoms.positions + self.dt * v
        self.calc.calculate(atoms, task=self.task)
        self.forces = np.asarray(self.calc.results["forces"], dtype=np.float64)
        self.stress = self._stress()
        atoms.velocities = atoms.velocities + 0.5 * self.dt * self.forces / m
        self.nsteps += 1

    def pressure_components(self) -> np.ndarray:
        """P_a = -sigma_aa + K_aa / V in eV/A^3 (ase's ``get_stress(include_ideal_gas=True)``, diagonal, negated)."""
        m = self.atoms.get_masses()[:, None]
        k = (m * self.atoms.velocities**2).sum(axis=0)
        return -np.diag(self.stress) + k / self.atoms.get_volume()

    def run(self, steps: int) -> list[dict]:
        log = []
        for _ in range(steps):
            self.step()
            entry = {"step": self.nsteps, "e_pot": self.potential_energy(), "e_kin": self.kinetic_energy(),
                     "temperature": self.temperature()}
            if self.barostat is not None:
                entry["volume"] = self.atoms.get_volume()
                entry["pressure"] = float(self.pressure_components().mean()) / GPA
            log.append(entry)
        return log


class Inhomogeneous_NPTBerendsen(NVTBerendsen):  # noqa: N801  (ASE's name)
    """Berendsen NPT with one scale per lattice vector (ASE's ``Inhomogeneous_NPTBerendsen``, dynamics.py:671-691):
    mu_a = 1 - dt beta / (3 tau_p) (P0 - P_a) mask_a, row a of the cell times mu_a, so the angles are kept.
    The step is the one of :class:`NVTBerendsen`; the forces of the previous call are used after the cell is scaled
    (one model call per step, as ``DeviceMD``; ASE calls the model again there)."""

    barostat = "inhomogeneous"

    def __init__(self, atoms, calculator, timestep: float = 2.0, temperature: float = 300.0, pressure: float = 1.01325e-4,
                 taut: float | None = None, taup: float | None = None, bulk_modulus: float | None = None,
                 fix_com: bool = True, mask=(1, 1, 1), task: PredTask | None = None) -> None:
        if bulk_modulus is None:
            raise ValueError("npt needs bulk_modulus (GPa)")
        self.target_pressure = float(pressure) * GPA
        beta = 1.0 / (float(bulk_modulus) * GPA)
        self.taupscl = (timestep * FS) / ((1000.0 * timestep if taup is None else taup) * FS) * beta / 3.0
        self.mask = np.asarray(mask, dtype=np.float64)
        super().__init__(atoms, calculator, timestep=timestep, temperature=temperature, taut=taut, fix_com=fix_com, task=task)

    def mu(self) -> np.ndarray:
        return 1.0 - self.taupscl * (self.target_pressure - self.pressure_components()) * self.mask

    def scale_cell(self) -> None:
        self.atoms.set_cell(self.mu()[:, None] * self.atoms.cell, scale_atoms=True)


class NPTBerendsen(Inhomogeneous_NPTBerendsen):
    """Isotropic Berendsen NPT (ASE's ``NPTBerendsen``, dynamics.py:693-715): mu = 1 - dt beta / (3 tau_p)
    (P0 - tr P / 3), the whole cell times mu, so its shape is kept."""

    barostat = "isotropic"

    def __init__(self, atoms, calculator, timestep: float = 2.0, temperature: float = 300.0, pressure: float = 1.01325e-4,
                 taut: float | None = None, taup: float | None = None, bulk_modulus: float | None = None,
                 fix_com: bool = True, task: PredTask | None = None) -> None:
        super().__init__(atoms, calculator, timestep=timestep, temperature=temperature, pressure=pressure, taut=taut, taup=taup,
                         bulk_modulus=bulk_modulus, fix_com=fix_com, task=task)

    def mu(self) -> np.ndarray:
        return np.full(3, 1.0 - self.taupscl * (self.target_pressure - self.pressure_components().sum() / 3.0))

    def scale_cell(self) -> None:
        self.atoms.set_cell(self.mu()[0] * self.atoms.cell, scale_atoms=True)


def fire_relax(atoms, calculator: CHGNetCalculator, fmax: float = 0.1, steps: int = 500, dt: float = 0.1,
               dt_max: float = 1.0, task: PredTask = "ef") -> dict:
    """Atomic-position relaxation with FIRE (Bitzek et al. 2006; the reference's default optimizer,
    dynamics.py:190-204), fixed cell.  Returns the trajectory of energies and the final max force."""
    n_min, f_inc, f_dec, alpha_start, f_alpha = 5, 1.1, 0.5, 0.1, 0.99
    v = np.zeros_like(atoms.positions)
    alpha, n_pos = alpha_start, 0
    energies = []
    for step in range(steps):
        calculator.calculate(atoms, task=task)
        f = np.asarray(calculator.results["forces"], dtype=np.float64)
        energies.append(float(calculator.results["energy"]))
        fnorm = float(np.sqrt((f**2).sum(axis=1)).max())
        if fnorm < fmax:
            break
        power = float((f * v).sum())
        if power > 0:
            v = (1 - alpha) * v + alpha * f * np.linalg.norm(v) / max(np.linalg.norm(f), 1e-30)
            n_pos += 1
            if n_pos > n_min:
                dt, alpha = min(dt * f_inc, dt_max), alpha * f_alpha
        else:
            v[:] = 0.0
            dt, alpha, n_pos = dt * f_dec, alpha_start, 0
        v = v + dt * f
        dr = dt * v
        norm = np.sqrt((dr**2).sum(axis=1)).max()
        if norm > 0.2:  # ase's maxstep
            dr *= 0.2 / norm
        atoms.positions = atoms.positions + dr
    return {"energies": energies, "fmax": fnorm, "steps": step + 1, "converged": fnorm < fmax}
