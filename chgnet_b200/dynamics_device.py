"""MD / relaxation with the whole step on the device (SURVEY.md §8 row f2).

The reference's MD loop is ``ase.md`` driving ``CHGNetCalculator.calculate`` (reference chgnet/model/dynamics.py:
129-181): every step converts the ASE atoms to a pymatgen ``Structure``, rebuilds the ``CrystalGraph`` on the CPU
(dynamics.py:156-157), copies it to the GPU, runs the model and copies energy / forces / stress back.  Here positions,
velocities and forces never leave the device:

* ``DeviceGraphBuilder`` (csrc/graph_device.cu) rebuilds the neighbour list / bond graph on the GPU.  Two policies:
  ``skin = 0`` - rebuild every step between the drift and the model call, exact cutoffs (the right choice for large
  cells: the build costs 0.5 ms for 10,000 atoms while a skin inflates the model's work, angles grow like (3 + skin)^6);
  ``skin > 0`` - a Verlet SKIN: the lists are built with cutoffs ``r + skin`` and reused until some atom has moved more
  than ``skin / 2`` since the last build, which lets the whole step be ONE CUDA graph replay (the right choice for small
  cells, where the ~140 launches of a step cost more than the kernels).  ``skin=None`` picks by the number of atoms.  Pairs beyond the model's cutoffs contribute exactly zero - CHGNet's polynomial envelope and hence the
  bond weights w_ag / w_bg vanish for d >= r_c (reference basis.py:184-205, layers.py:118-126, 245-254) - so the skin
  changes no result (tests/test_dynamics_device_gpu.py compares against rebuilding every step);
* between rebuilds the step = [half kick + drift] -> ``chg_forward`` -> [half kick] is ONE CUDA graph replay
  (captured after every rebuild): ~140 kernel launches become one;
* the host reads one double per step (the skin test) and, when asked, the energies.

``DeviceMD`` = velocity Verlet (NVE, what ``ase.md.verlet.VelocityVerlet`` does) or Berendsen NVT / NPT (ASE's
``NVTBerendsen``, ``Inhomogeneous_NPTBerendsen``, ``NPTBerendsen``: the reference's ``MolecularDynamics`` ensembles) with
the cell in device memory; ``DeviceFIRE`` = FIRE relaxation at fixed cell with its state on the device.  The host
drivers of ``chgnet_b200.dynamics`` are the checkers.  Under a changing cell the skin test is ``verlet_lists_valid``
(displacement in the build-time frame plus the strain of the cell).
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

from chgnet_b200._lib import ChgnetB200Error, load_library
from chgnet_b200.dynamics import ATOMIC_MASSES, FS, GPA, KB
from chgnet_b200.graph_device import DeviceGraphBuilder

_LIB = None

# chg_md_* flags (include/chgnet_b200.h) and offsets into the 64-double cell state
_THERMO, _BARO_ISO, _BARO_ANISO, _FIX_COM = 1, 2, 4, 8
_BARO = _BARO_ISO | _BARO_ANISO
_CS_DOUBLES, _CS_L, _CS_LINV, _CS_LOLD_INV, _CS_LREF, _CS_VOL, _CS_D2 = 64, 0, 9, 18, 27, 45, 52
_THERMOSTAT_MSG = "Thermostat not supported, choose in 'Nose-Hoover', 'Berendsen', 'Berendsen_inhomogeneous'"


def ensemble_flags(ensemble: str, thermostat: str, bulk_modulus: float | None) -> int:
    """The reference's ``MolecularDynamics`` choices (dynamics.py:578-720) -> chg_md_* flags (0 = NVE)."""
    ens, th = str(ensemble).lower(), str(thermostat).lower()
    if ens == "nve":
        return 0
    if ens not in ("nvt", "npt"):
        raise ValueError(f"Ensemble {ensemble!r} not supported, choose in 'nve', 'nvt', 'npt'")
    if th == "nose-hoover":
        raise NotImplementedError("Nose-Hoover (ASE's NPT) is not implemented by DeviceMD; use thermostat='Berendsen_inhomogeneous' "
                                  "(nvt / npt) or 'npt_berendsen' (npt)")
    if ens == "nvt":
        if th.startswith("berendsen"):
            return _THERMO
        raise ValueError(_THERMOSTAT_MSG)
    if th == "berendsen_inhomogeneous":
        baro = _BARO_ANISO
    elif th == "npt_berendsen":
        baro = _BARO_ISO
    else:
        raise ValueError(_THERMOSTAT_MSG)
    if bulk_modulus is None:
        raise ValueError("npt needs bulk_modulus (GPa): it sets the barostat's compressibility, and fitting it by an equation "
                         "of state would need a variable-cell relaxation")
    return _THERMO | baro


def verlet_lists_valid(d: float, eps: float, cutoff: float, skin: float) -> bool:
    """May neighbour lists built with ``cutoff + skin`` still be used for ``cutoff``?

    ``d`` = max_i |(s_i - s_ref,i) L_ref| is the largest displacement since the build, measured in the build-time
    frame; ``eps`` = ||L_ref^-1 L - I||_F is the strain of the cell since then.  A pair farther than ``cutoff + skin``
    at the build is now at least (|r_0| - 2d) sigma_min(L_ref^-1 L) >= (cutoff + skin - 2d)(1 - eps) apart, so the
    lists are complete while that is >= ``cutoff``.  Written as 2d <= skin - eps (cutoff + skin - 2d), which for
    eps = 0 is exactly d <= skin / 2 (the test of a fixed cell).  NaN never passes."""
    two_d = 2.0 * d
    return two_d <= skin and two_d <= skin - eps * (cutoff + skin - two_d)


def _lib():
    global _LIB
    if _LIB is None:
        lib = load_library()
        P, I, D = ctypes.c_void_p, ctypes.c_int32, ctypes.c_double
        lib.chg_md_kick_drift.restype = I
        lib.chg_md_kick_drift.argtypes = [P, P, P, P, I, D, P, P, P, P, P, P]
        lib.chg_md_kick.restype = I
        lib.chg_md_kick.argtypes = [P, P, P, I, D, P, P]
        lib.chg_fire_step.restype = I
        lib.chg_fire_step.argtypes = [P, P, P, I, P, P, P, P, D, D, P]
        _LIB = lib
    return _LIB


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise ChgnetB200Error(f"{what} failed ({rc}): {_lib().chg_last_error().decode()}")


class _DeviceSystem:
    """Positions / velocities / forces on the device + the model evaluation with a skin-managed graph."""

    def __init__(self, model, numbers, positions, cell, *, skin: float | None = 0.5, use_cuda_graph: bool = True) -> None:
        self.model = model.eval()
        self.dev = model.device
        if self.dev.type != "cuda":
            raise ChgnetB200Error("device MD needs the model on a CUDA device")
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        self.numbers = np.asarray(numbers, dtype=np.int64).reshape(-1)
        self.n = len(self.numbers)
        self.lattice = np.asarray(cell, dtype=np.float64).reshape(3, 3)  # host copy: the cell of the last list build
        self.inv_cell = np.ascontiguousarray(np.linalg.inv(self.lattice))
        f64 = dict(dtype=torch.float64, device=self.dev)
        self.x = torch.as_tensor(np.asarray(positions, dtype=np.float64).reshape(-1, 3)).to(self.dev).contiguous()
        self.v = torch.zeros(self.n, 3, **f64)
        self.f = torch.zeros(self.n, 3, **f64)
        self.inv_mass = torch.as_tensor(1.0 / ATOMIC_MASSES[self.numbers - 1]).to(self.dev)
        self.frac64 = torch.empty(self.n, 3, **f64)
        self.frac32 = torch.empty(self.n, 3, dtype=torch.float32, device=self.dev)
        self.x_ref = self.x.clone()
        self.max_disp2 = torch.zeros(1, **f64)
        self.e_kin = torch.zeros(1, **f64)
        if skin is None:  # large cells: exact lists every step; small cells: skin + one CUDA graph per step
            skin = 0.0 if self.n >= 2000 else 0.5
        self.skin = float(skin)
        if self.skin < 0.0:
            raise ValueError("skin must be >= 0")
        self.every_step = self.skin == 0.0
        gc = model.graph_converter
        self.builder = DeviceGraphBuilder(self.dev, float(gc.atom_graph_cutoff) + self.skin, float(gc.bond_graph_cutoff) + self.skin)
        self.compact = not model._arch.get("mlp_out_bias", False)
        self.use_cuda_graph = use_cuda_graph and not self.every_step
        self.batch = None
        self.graph = None
        self.out: dict | None = None
        self.n_builds = 0
        self.n_steps = 0
        self.n_captures = 0
        self.t_rebuild = self.t_capture = 0.0  # host seconds spent rebuilding lists / capturing step graphs
        self._init_state()
        self._update_frac()
        self._rebuild()
        self._forward()
        self._old_graph = None

    # ---- pieces ---------------------------------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _init_state(self) -> None:
        """Extra device state of a subclass, allocated before the first list build."""

    def _update_frac(self) -> None:
        fr = self.x @ torch.as_tensor(self.inv_cell).to(self.dev)
        self.frac64.copy_(fr)
        self.frac32.copy_(fr.to(torch.float32))

    def _rebuild(self) -> None:
        """New neighbour lists (cutoffs + skin) from the current positions; the captured step graph is dropped."""
        batch = self.builder.build_batch(self.numbers, self.frac64, self.lattice, with_reverse=True, compact_bonds=self.compact)
        batch.frac = self.frac32  # the model reads the positions the integrator writes
        self.batch = batch
        self.x_ref.copy_(self.x)
        self.max_disp2.zero_()
        self._old_graph, self.graph = self.graph, None  # keep the pool's last user alive until the next capture
        self.n_builds += 1

    def _forward(self) -> None:
        nat = self.model._get_native()
        self.out = nat(self.batch, need_grad=True)
        self.f.copy_(self.out["force"])

    def needs_rebuild(self) -> bool:
        """One double from the device: has some atom moved more than skin / 2 since the lists were built?"""
        return float(self.max_disp2.item()) > (0.5 * self.skin) ** 2

    @property
    def potential_energy(self) -> float:
        return float((self.out["energy"] + self.out["e_ref"])[0].item())

    def positions(self) -> np.ndarray:
        return self.x.cpu().numpy()


class DeviceMD(_DeviceSystem):
    """Molecular dynamics with positions, velocities, forces and the cell resident on the device; ``timestep`` in fs.

    The keywords follow the reference's ``MolecularDynamics`` (dynamics.py:433-715): ``ensemble`` "nve" (velocity
    Verlet), "nvt" (``thermostat`` "Berendsen" or "Berendsen_inhomogeneous": ASE's ``NVTBerendsen``) or "npt"
    (``thermostat`` "Berendsen_inhomogeneous": ASE's ``Inhomogeneous_NPTBerendsen``, every lattice vector scaled by its
    own diagonal pressure so the cell angles are kept; "npt_berendsen": the isotropic ``NPTBerendsen``).
    ``temperature`` in K, ``pressure`` and ``bulk_modulus`` in GPa, ``taut`` / ``taup`` in fs (default 100 and 1000
    timesteps).  ``fix_com`` removes the mean momentum every nvt / npt step (ASE's ``fixcm``); ``mask`` switches the
    per-axis barostat off along lattice vectors.

    The step is the one of ASE's Berendsen classes with ONE model call: ASE evaluates the forces again after rescaling
    the cell (``set_cell(scale_atoms=True)``); this driver keeps the forces of the previous call, as LAMMPS' ``fix
    press/berendsen`` does.  The difference per step is of order ``|mu - 1| |F|`` (``|mu - 1|`` ~ 3e-6 at the default
    couplings, 1 GPa off target and B = 100 GPa).  The cell, the targets and the couplings live in device buffers,
    so with a skin the step stays one CUDA graph replay, and ``set_target`` changes the targets without a new capture.
    The host checkers ``chgnet_b200.dynamics.NVTBerendsen`` / ``NPTBerendsen`` / ``Inhomogeneous_NPTBerendsen`` follow
    the same sequence."""

    def __init__(self, model, numbers, positions, cell, *, timestep: float = 2.0, velocities=None, skin: float | None = None,
                 use_cuda_graph: bool = True, ensemble: str = "nve", thermostat: str = "Berendsen_inhomogeneous",
                 temperature: float = 300.0, pressure: float = 1.01325e-4, taut: float | None = None,
                 taup: float | None = None, bulk_modulus: float | None = None, fix_com: bool = True, mask=(1, 1, 1)) -> None:
        self.flags = ensemble_flags(ensemble, thermostat, bulk_modulus)
        self.ensemble = str(ensemble).lower()
        self.timestep = float(timestep)
        self.taut = 100.0 * self.timestep if taut is None else float(taut)
        self.taup = 1000.0 * self.timestep if taup is None else float(taup)
        self.bulk_modulus = None if bulk_modulus is None else float(bulk_modulus)
        if self.flags and not self.taut > 0.0:
            raise ValueError("taut must be > 0")
        if self.flags & _BARO and not (self.taup > 0.0 and self.bulk_modulus > 0.0):
            raise ValueError("taup and bulk_modulus must be > 0")
        self.mask = tuple(float(m) for m in mask)
        if len(self.mask) != 3:
            raise ValueError("mask needs three entries, one per lattice vector")
        if self.flags and fix_com:
            self.flags |= _FIX_COM
        self.target_temperature, self.target_pressure = float(temperature), float(pressure)
        self.n_strain_builds = 0  # rebuilds that the displacement alone would not have triggered
        super().__init__(model, numbers, positions, cell, skin=skin, use_cuda_graph=use_cuda_graph)
        gc = model.graph_converter
        self.r_list = max(float(gc.atom_graph_cutoff), float(gc.bond_graph_cutoff))
        self.dt = float(timestep) * FS
        if self.flags:
            self._write_params()
        if velocities is not None:
            self.v.copy_(torch.as_tensor(np.asarray(velocities, dtype=np.float64)).to(self.dev))
        self._refresh_kinetic()

    # ---- device state of the Berendsen ensembles --------------------------------------------------------------------
    def _init_state(self) -> None:
        if not self.flags:
            return
        f64 = dict(dtype=torch.float64, device=self.dev)
        inv = np.linalg.inv(self.lattice)
        cs = np.zeros(_CS_DOUBLES)
        cs[_CS_L:_CS_L + 9], cs[_CS_LINV:_CS_LINV + 9], cs[_CS_LOLD_INV:_CS_LOLD_INV + 9] = self.lattice.ravel(), inv.ravel(), inv.ravel()
        cs[_CS_VOL] = abs(np.linalg.det(self.lattice))
        self.cs = torch.as_tensor(cs).to(self.dev)
        self.params = torch.zeros(8, **f64)
        nblk = int(_lib().chg_md_partial_blocks(self.n))
        self.k_part = torch.zeros(nblk, 4, **f64)
        self.mom_part = torch.zeros(nblk, 3, **f64)
        self.virial = torch.zeros(9, **f64)
        self.lat32 = torch.as_tensor(self.lattice.reshape(1, 9), dtype=torch.float32).to(self.dev)
        self.s_ref = torch.zeros(self.n, 3, **f64)

    def _write_params(self) -> None:
        beta = 0.0 if self.bulk_modulus is None else 1.0 / (self.bulk_modulus * GPA)
        dt, taut, taup = self.timestep * FS, self.taut * FS, self.taup * FS
        p = [self.target_temperature, self.target_pressure * GPA, dt / taut, dt / taup * beta / 3.0, *self.mask, KB]
        self.params.copy_(torch.tensor(p, dtype=torch.float64))  # stream-ordered: the next step reads the new targets

    def set_target(self, temperature: float | None = None, pressure: float | None = None) -> None:
        """New thermostat / barostat targets (K, GPa) from the next step on; the captured step graph is kept."""
        if not self.flags:
            raise ValueError("set_target needs ensemble='nvt' or 'npt'")
        if temperature is not None:
            self.target_temperature = float(temperature)
        if pressure is not None:
            self.target_pressure = float(pressure)
        self._write_params()

    def _refresh_kinetic(self) -> None:
        """Kinetic energy of the current velocities (the thermostat of the next step reads it)."""
        lib, st = _lib(), self._stream()
        with torch.cuda.device(self.dev):
            if self.flags:
                _check(lib.chg_md_kick_partials(self.v.data_ptr(), None, self.inv_mass.data_ptr(), self.n, 0.0, self.k_part.data_ptr(), st),
                       "chg_md_kick_partials")
            else:  # a kick of length zero leaves v as it is and sums the kinetic energy
                self.e_kin.zero_()
                _check(lib.chg_md_kick(self.v.data_ptr(), self.f.data_ptr(), self.inv_mass.data_ptr(), self.n, 0.0, self.e_kin.data_ptr(), st),
                       "chg_md_kick")

    def _rebuild(self) -> None:
        if not self.flags:
            super()._rebuild()
            return
        self.lattice = self.cs[_CS_L:_CS_L + 9].cpu().numpy().reshape(3, 3)
        batch = self.builder.build_batch(self.numbers, self.frac64, self.lattice, with_reverse=True, compact_bonds=self.compact)
        batch.frac = self.frac32  # the model reads the positions and the cell the integrator writes
        batch.lattice = self.lat32
        self.batch = batch
        self.s_ref.copy_(self.frac64)
        self.cs[_CS_LREF:_CS_LREF + 18].copy_(self.cs[_CS_L:_CS_L + 18])  # L_ref, L_ref^-1 <- L, L^-1
        self.cs[_CS_D2:_CS_D2 + 2].zero_()
        self._old_graph, self.graph = self.graph, None
        self.n_builds += 1

    def _forward(self) -> None:
        super()._forward()
        if self.flags & _BARO:
            self.virial.copy_(self.out["virial"][0])

    def needs_rebuild(self) -> bool:
        if not self.flags:
            return super().needs_rebuild()
        d2, eps = self.cs[_CS_D2:_CS_D2 + 2].tolist()  # one small read per step
        d = math.sqrt(d2)
        if verlet_lists_valid(d, eps, self.r_list, self.skin):
            return False
        if 2.0 * d <= self.skin:
            self.n_strain_builds += 1
        return True

    def _carried(self) -> tuple:
        """The device tensors one step reads and writes (saved around the warm-up step of a capture)."""
        if not self.flags:
            return (self.x, self.v, self.f, self.max_disp2)
        return (self.x, self.v, self.f, self.virial, self.cs, self.k_part, self.lat32)

    # ---- public -------------------------------------------------------------------------------------------------------
    def set_temperature(self, kelvin: float, seed: int = 0) -> None:
        rng = np.random.default_rng(seed)
        m = ATOMIC_MASSES[self.numbers - 1][:, None]
        v = rng.normal(size=(self.n, 3)) * np.sqrt(KB * kelvin / m)
        v -= (m * v).sum(axis=0) / m.sum()
        self.v.copy_(torch.as_tensor(v).to(self.dev))
        self._refresh_kinetic()

    def _step_body(self) -> None:
        if self.flags:
            self._step_body_berendsen()
            return
        lib, st = _lib(), self._stream()
        with torch.cuda.device(self.dev):
            _check(lib.chg_md_kick_drift(self.x.data_ptr(), self.v.data_ptr(), self.f.data_ptr(), self.inv_mass.data_ptr(), self.n, self.dt,
                                         self.inv_cell.ctypes.data, self.frac64.data_ptr(), self.frac32.data_ptr(),
                                         self.x_ref.data_ptr(), self.max_disp2.data_ptr(), st), "chg_md_kick_drift")
        if self.every_step:  # exact neighbour lists for the new positions (0.5 ms for 10,000 atoms)
            self._rebuild()
        self._forward()
        self.e_kin.zero_()
        with torch.cuda.device(self.dev):
            _check(lib.chg_md_kick(self.v.data_ptr(), self.f.data_ptr(), self.inv_mass.data_ptr(), self.n, self.dt, self.e_kin.data_ptr(),
                                   self._stream()), "chg_md_kick")

    def _step_body_berendsen(self) -> None:
        """[thermostat, barostat, cell] -> [scale + kick, mean momentum + drift] -> chg_forward -> [kick + K partials]."""
        lib, st = _lib(), self._stream()
        with torch.cuda.device(self.dev):
            _check(lib.chg_md_cell_step(self.params.data_ptr(), self.cs.data_ptr(), self.k_part.data_ptr(), self.n,
                                        self.virial.data_ptr(), self.lat32.data_ptr(), self.flags, st), "chg_md_cell_step")
            _check(lib.chg_md_kick_drift_cell(self.x.data_ptr(), self.v.data_ptr(), self.f.data_ptr(), self.inv_mass.data_ptr(), self.n,
                                              self.dt, self.cs.data_ptr(), self.mom_part.data_ptr(), self.frac64.data_ptr(),
                                              self.frac32.data_ptr(), None if self.every_step else self.s_ref.data_ptr(), self.flags, st),
                   "chg_md_kick_drift_cell")
        if self.every_step:
            self._rebuild()
        self._forward()
        with torch.cuda.device(self.dev):
            _check(lib.chg_md_kick_partials(self.v.data_ptr(), self.f.data_ptr(), self.inv_mass.data_ptr(), self.n, self.dt,
                                            self.k_part.data_ptr(), self._stream()), "chg_md_kick_partials")

    def step(self) -> None:
        if self.use_cuda_graph:
            if self.graph is None:
                self._capture()
            self.graph.replay()
        else:
            self._step_body()
        self.n_steps += 1
        if not self.every_step and self.needs_rebuild():
            import time

            t0 = time.perf_counter()
            self._rebuild()
            self.t_rebuild += time.perf_counter() - t0

    def _capture(self) -> None:
        """Capture one step for the current topology.  Raw capture_begin / capture_end
        on a side stream with one memory pool shared by all captures of this run (``torch.cuda.graph`` would run the
        garbage collector and empty the allocator cache at every capture)."""
        import time

        t0 = time.perf_counter()
        nat = self.model._get_native()
        nat.reserve(self.batch, need_grad=True)  # never reallocate the workspace inside a capture
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(self.dev)
            self._pool = torch.cuda.graph_pool_handle()
        s = self._side
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            if not getattr(self, "_warmed", False):
                # once: a real step on the side stream (lazily set kernel attributes, allocator warm-up), then undone
                state = [t.clone() for t in self._carried()]
                self._step_body()
                s.synchronize()
                for t, saved in zip(self._carried(), state):
                    t.copy_(saved)
                self._warmed = True
            # the previous capture stays alive until the new one exists: the shared pool must never drop to zero users
            g = torch.cuda.CUDAGraph()
            g.capture_begin(pool=self._pool, capture_error_mode="thread_local")  # other threads (NCCL watchdog) may call CUDA
            try:
                self._step_body()
            finally:
                g.capture_end()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        self._old_graph = None
        self.graph = g  # capturing executed nothing: the state is still the pre-step state
        self.n_captures += 1
        self.t_capture += time.perf_counter() - t0

    @property
    def kinetic_energy(self) -> float:
        if self.flags:
            return 0.5 * float(self.k_part[:, 3].sum().item())
        return float(self.e_kin.item())

    def temperature(self) -> float:
        return 2.0 * self.kinetic_energy / (3.0 * self.n * KB)

    def cell(self) -> np.ndarray:
        """The current cell (rows = lattice vectors, A) as a host 3x3 array."""
        if self.flags:
            return self.cs[_CS_L:_CS_L + 9].cpu().numpy().reshape(3, 3)
        return self.lattice.copy()

    @property
    def volume(self) -> float:
        if self.flags:
            return float(self.cs[_CS_VOL].item())
        return abs(float(np.linalg.det(self.lattice)))

    def pressure(self) -> float:
        """Pressure in GPa with the ideal-gas term, (2 E_kin - tr virial) / (3 V): what the barostat controls."""
        tr = float(self.out["virial"][0, [0, 4, 8]].sum().item())
        return (2.0 * self.kinetic_energy - tr) / (3.0 * self.volume) / GPA

    def run(self, steps: int, log_every: int = 1) -> list[dict]:
        log = []
        for i in range(steps):
            self.step()
            if log_every and (i + 1) % log_every == 0:
                entry = {"step": self.n_steps, "e_pot": self.potential_energy, "e_kin": self.kinetic_energy,
                         "temperature": self.temperature()}
                if self.flags & _BARO:
                    entry["volume"], entry["pressure"] = self.volume, self.pressure()
                log.append(entry)
        return log


class DeviceFIRE(_DeviceSystem):
    """FIRE relaxation at fixed cell (the reference's default optimizer, dynamics.py:190-204) with the optimizer state
    on the device; the host looks at the largest force every ``check_every`` steps."""

    def __init__(self, model, numbers, positions, cell, *, dt: float = 0.1, dt_max: float = 1.0, max_step: float = 0.2,
                 skin: float | None = None) -> None:
        super().__init__(model, numbers, positions, cell, skin=skin, use_cuda_graph=False)
        self.dt_max, self.max_step = float(dt_max), float(max_step)
        self.state = torch.zeros(12, dtype=torch.float64, device=self.dev)
        self.state[0], self.state[1] = dt, 0.1

    def run(self, fmax: float = 0.1, steps: int = 500, check_every: int = 5) -> dict:
        lib = _lib()
        energies = []
        fm = float(self.f.pow(2).sum(dim=1).max().sqrt().item())
        it = 0
        while it < steps and fm >= fmax:
            with torch.cuda.device(self.dev):
                _check(lib.chg_fire_step(self.x.data_ptr(), self.v.data_ptr(), self.f.data_ptr(), self.n, self.state.data_ptr(),
                                         self.inv_cell.ctypes.data, self.frac64.data_ptr(), self.frac32.data_ptr(), self.dt_max,
                                         self.max_step, self._stream()), "chg_fire_step")
            # skin test on the host side of the loop (positions moved by at most max_step)
            if self.every_step:
                self._rebuild()
            else:
                d2 = float(((self.x - self.x_ref) ** 2).sum(dim=1).max().item())
                if d2 > (0.5 * self.skin) ** 2:
                    self._rebuild()
            self._forward()
            it += 1
            if it % check_every == 0 or it == steps:
                fm = float(self.f.pow(2).sum(dim=1).max().sqrt().item())
                energies.append(self.potential_energy)
        return {"energies": energies, "fmax": fm, "steps": it, "converged": fm < fmax, "graph_builds": self.n_builds}


__all__ = ["DeviceMD", "DeviceFIRE", "ensemble_flags", "verlet_lists_valid"]
