"""CPU: the strain-aware Verlet-skin test of DeviceMD (chgnet_b200.dynamics_device.verlet_lists_valid) against brute-force
neighbour lists over periodic images, and the host Berendsen checkers of chgnet_b200.dynamics (ASE's NVTBerendsen,
NPTBerendsen and Inhomogeneous_NPTBerendsen restated) driven by a small numpy pair potential."""
import itertools

import numpy as np
import pytest

from chgnet_b200.dynamics import (FS, GPA, KB, Atoms, Inhomogeneous_NPTBerendsen, NPTBerendsen, NVTBerendsen,
                                  berendsen_lambda)
from chgnet_b200.dynamics_device import ensemble_flags, verlet_lists_valid


# ---- rebuild criterion ----------------------------------------------------------------------------------------------
def _pairs(frac, lat, rc):
    """{(i, j, image)} with |(s_j + image - s_i) L| < rc, every periodic image that can be in range."""
    inv = np.linalg.inv(lat)
    reach = [int(np.ceil(rc * np.linalg.norm(inv[:, a]))) + 1 for a in range(3)]
    out = set()
    for img in itertools.product(*(range(-r, r + 1) for r in reach)):
        d = (frac[None, :, :] + np.asarray(img, dtype=np.float64)[None, None, :] - frac[:, None, :]) @ lat
        ii, jj = np.nonzero((d**2).sum(axis=-1) < rc * rc)
        out.update((int(i), int(j), img) for i, j in zip(ii, jj) if not (i == j and img == (0, 0, 0)))
    return out


def _random_cell(rng):
    lat = np.diag(rng.uniform(4.5, 7.0, 3)) + np.triu(rng.uniform(-1.5, 1.5, (3, 3)), 1)
    return lat[rng.permutation(3)][:, rng.permutation(3)] if rng.random() < 0.3 else lat


def test_rebuild_criterion_keeps_every_pair_within_the_cutoff():
    rng = np.random.default_rng(11)
    r, kept, rejected = 3.0, 0, 0
    for trial in range(160):
        lat_ref = _random_cell(rng)
        n = int(rng.integers(4, 17))
        s_ref = rng.random((n, 3))
        skin = float(rng.choice([0.3, 0.5, 0.8]))
        lists = _pairs(s_ref, lat_ref, r + skin)
        # displacement in the build frame and a deformation of the cell, sized around the criterion's edge
        disp = rng.normal(size=(n, 3)) * rng.uniform(0.0, 0.25) * skin
        strain = rng.normal(size=(3, 3)) * rng.uniform(0.0, 0.06)
        a = np.eye(3) + strain
        lat = lat_ref @ a
        s = s_ref + disp @ np.linalg.inv(lat_ref)
        d = float(np.sqrt((((s - s_ref) @ lat_ref) ** 2).sum(axis=1)).max())
        eps = float(np.linalg.norm(np.linalg.inv(lat_ref) @ lat - np.eye(3)))
        if verlet_lists_valid(d, eps, r, skin):
            kept += 1
            missing = _pairs(s, lat, r) - lists
            assert not missing, (trial, d, eps, sorted(missing)[:5])
        else:
            rejected += 1
    assert kept >= 30 and rejected >= 30, (kept, rejected)


def test_strain_term_catches_what_the_displacement_test_misses():
    # no atom moves in the build frame, but the cell shrinks by 15 %: a pair just beyond r + skin comes within r
    r, skin = 3.0, 0.5
    lat_ref = np.diag([10.0, 10.0, 10.0])
    s_ref = np.array([[0.0, 0.0, 0.0], [(r + skin + 0.01) / 10.0, 0.0, 0.0]])
    lists = _pairs(s_ref, lat_ref, r + skin)
    lat = 0.85 * lat_ref
    assert _pairs(s_ref, lat, r) - lists  # the old lists really are incomplete
    eps = float(np.linalg.norm(np.linalg.inv(lat_ref) @ lat - np.eye(3)))
    assert verlet_lists_valid(0.0, 0.0, r, skin) and not verlet_lists_valid(0.0, eps, r, skin)


def test_rebuild_criterion_without_strain_is_the_fixed_cell_test():
    rng = np.random.default_rng(5)
    for r in (3.0, 5.0, 6.0, 6.3):
        for skin in (0.1, 0.3, 0.5, 1.2):
            half = skin / 2
            ds = list(rng.uniform(0.0, skin, 200)) + [0.0, half, np.nextafter(half, 0.0), np.nextafter(half, 1.0), skin, 1e-300]
            for d in ds:
                assert verlet_lists_valid(float(d), 0.0, r, skin) == (d <= skin / 2), (r, skin, d)
    assert not verlet_lists_valid(float("nan"), 0.0, 6.0, 0.5)
    assert not verlet_lists_valid(0.0, float("nan"), 6.0, 0.5)
    assert not verlet_lists_valid(0.0, 1.5, 6.0, 0.5)


def test_ensemble_choices_follow_the_reference():
    assert ensemble_flags("nve", "anything", None) == 0
    assert ensemble_flags("NVT", "Berendsen", None) == ensemble_flags("nvt", "Berendsen_inhomogeneous", None) == 1
    assert ensemble_flags("npt", "Berendsen_inhomogeneous", 100.0) == 1 | 4
    assert ensemble_flags("npt", "npt_berendsen", 100.0) == 1 | 2
    with pytest.raises(ValueError, match="Thermostat not supported"):
        ensemble_flags("nvt", "Langevin", None)
    with pytest.raises(ValueError, match="Thermostat not supported"):
        ensemble_flags("npt", "Berendsen", 100.0)
    with pytest.raises(ValueError, match="Ensemble"):
        ensemble_flags("nph", "Berendsen", None)
    for ens in ("nvt", "npt"):
        with pytest.raises(NotImplementedError, match="Nose-Hoover"):
            ensemble_flags(ens, "Nose-Hoover", 100.0)
    with pytest.raises(ValueError, match="bulk_modulus"):
        ensemble_flags("npt", "Berendsen_inhomogeneous", None)


# ---- host integrators -----------------------------------------------------------------------------------------------
class PairCalc:
    """Morse pair potential over periodic images: energy (eV), forces (eV/A), stress = (1/V) dE/d(strain) (eV/A^3),
    the sign convention of CHGNetCalculator."""

    def __init__(self, depth=0.3, a=1.2, r0=3.0, rc=5.0):
        self.depth, self.a, self.r0, self.rc = depth, a, r0, rc
        self.results = {}

    def calculate(self, atoms, task="efs"):
        lat, x = atoms.cell, atoms.positions
        frac = x @ np.linalg.inv(lat)
        n = len(x)
        e, f, w = 0.0, np.zeros((n, 3)), np.zeros((3, 3))
        inv = np.linalg.inv(lat)
        reach = [int(np.ceil(self.rc * np.linalg.norm(inv[:, k]))) + 1 for k in range(3)]
        for img in itertools.product(*(range(-r, r + 1) for r in reach)):
            rv = (frac[None, :, :] + np.asarray(img, dtype=np.float64) - frac[:, None, :]) @ lat  # r_j - r_i
            dist = np.sqrt((rv**2).sum(axis=-1))
            ok = (dist < self.rc) & (dist > 1e-9)
            ex = np.exp(-self.a * (dist - self.r0))
            phi = self.depth * ((1 - ex) ** 2 - 1)
            dphi = 2 * self.depth * self.a * (1 - ex) * ex
            e += 0.5 * phi[ok].sum()
            g = np.where(ok, dphi / np.where(ok, dist, 1.0), 0.0)[..., None] * rv  # dE/d r_ij on the pair (i, j)
            f += g.sum(axis=1)
            w += 0.5 * np.einsum("ija,ijb->ab", rv, g)
        self.results = {"energy": e, "forces": f, "stress": w / abs(np.linalg.det(lat))}


def _crystal(rng, scale=1.0, triclinic=True):
    base = np.array([[0, 0, 0], [0.5, 0.5, 0], [0.5, 0, 0.5], [0, 0.5, 0.5]], dtype=np.float64)
    cells = np.array(list(itertools.product(range(2), repeat=3)), dtype=np.float64)
    frac = ((base[None] + cells[:, None]) / 2.0).reshape(-1, 3)
    lat = np.diag([7.4, 7.3, 7.5]) * scale
    if triclinic:
        lat[1, 0], lat[2, 0], lat[2, 1] = 0.6, -0.4, 0.3
    x = frac @ lat + rng.normal(0.0, 0.05, frac.shape)
    return Atoms(np.full(len(frac), 29), x, lat)


def _angles_and_lengths(lat):
    ln = np.linalg.norm(lat, axis=1)
    cos = [lat[i] @ lat[j] / (ln[i] * ln[j]) for i, j in ((0, 1), (0, 2), (1, 2))]
    return ln, np.array(cos)


def test_lambda_is_clamped():
    assert berendsen_lambda(1000.0, 10.0, 0.5) == 0.9
    assert berendsen_lambda(10.0, 1000.0, 0.5) == 1.1
    assert berendsen_lambda(1000.0, 10.0, 3.0) == 0.9  # sqrt of a negative number in ASE's formula: clamped, not NaN
    assert berendsen_lambda(300.0, 300.0, 0.1) == 1.0
    assert abs(berendsen_lambda(300.0, 330.0, 0.02) - np.sqrt(1.002)) < 1e-15
    rng = np.random.default_rng(1)
    atoms = _crystal(rng)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 0.05
    hot = NVTBerendsen(atoms, PairCalc(), timestep=1.0, temperature=1.0, taut=1.0)
    hot.step()
    assert hot.last_lambda == 0.9
    atoms = _crystal(rng)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 1e-4
    cold = NVTBerendsen(atoms, PairCalc(), timestep=1.0, temperature=5000.0, taut=1.0)
    cold.step()
    assert cold.last_lambda == 1.1


def test_zero_temperature_gives_the_largest_scale_and_no_motion():
    atoms = _crystal(np.random.default_rng(2), triclinic=False)
    md = NVTBerendsen(atoms, PairCalc(depth=0.0), timestep=2.0, temperature=300.0)
    x0 = atoms.positions.copy()
    md.run(3)
    assert md.last_lambda == 1.1
    assert np.all(atoms.velocities == 0.0) and np.all(atoms.positions == x0)


def test_isotropic_barostat_keeps_the_cell_shape():
    rng = np.random.default_rng(3)
    atoms = _crystal(rng, scale=0.97)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 0.02
    ln0, cos0 = _angles_and_lengths(atoms.cell)
    md = NPTBerendsen(atoms, PairCalc(), timestep=2.0, temperature=300.0, pressure=0.0, taup=20.0, bulk_modulus=20.0)
    md.run(10)
    ln, cos = _angles_and_lengths(atoms.cell)
    assert abs(ln[0] / ln0[0] - 1.0) > 1e-4  # the cell did change
    assert np.abs(ln / ln[0] - ln0 / ln0[0]).max() < 1e-12 and np.abs(cos - cos0).max() < 1e-12


def test_inhomogeneous_barostat_keeps_the_angles_and_the_masked_vector():
    rng = np.random.default_rng(4)
    atoms = _crystal(rng, scale=0.97)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 0.02
    c0 = atoms.cell[2].copy()
    ln0, cos0 = _angles_and_lengths(atoms.cell)
    md = Inhomogeneous_NPTBerendsen(atoms, PairCalc(), timestep=2.0, pressure=0.0, taup=20.0, bulk_modulus=20.0, mask=(1, 1, 0))
    md.run(10)
    ln, cos = _angles_and_lengths(atoms.cell)
    assert np.abs(ln[:2] / ln0[:2] - 1.0).min() > 1e-4
    assert np.abs(cos - cos0).max() < 1e-12
    assert np.array_equal(atoms.cell[2], c0)


def test_scale_atoms_keeps_fractional_coordinates():
    rng = np.random.default_rng(5)
    atoms = _crystal(rng)
    frac0 = atoms.positions @ np.linalg.inv(atoms.cell)
    new = atoms.cell @ (np.eye(3) + rng.normal(size=(3, 3)) * 0.05)
    atoms.set_cell(new, scale_atoms=True)
    assert np.abs(atoms.positions @ np.linalg.inv(atoms.cell) - frac0).max() < 1e-12
    assert abs(atoms.get_volume() - abs(np.linalg.det(new))) < 1e-9
    kept = atoms.positions.copy()
    atoms.set_cell(new * 1.1)
    assert np.array_equal(atoms.positions, kept)


def test_fix_com_removes_the_total_momentum():
    rng = np.random.default_rng(6)
    atoms = _crystal(rng)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 0.03 + 0.01  # a drift of the centre of mass
    m = atoms.get_masses()[:, None]
    assert np.abs((m * atoms.velocities).sum(axis=0)).max() > 1.0
    md = Inhomogeneous_NPTBerendsen(atoms, PairCalc(), timestep=2.0, bulk_modulus=50.0)
    md.run(5)
    assert np.abs((m * atoms.velocities).sum(axis=0)).max() < 1e-12


def test_compressed_cell_expands_on_the_first_step():
    rng = np.random.default_rng(7)
    atoms = _crystal(rng, scale=0.9)
    calc = PairCalc()
    calc.calculate(atoms)
    assert -np.trace(calc.results["stress"]) / 3 > 0.1 * GPA  # compressed: positive pressure
    for cls in (NPTBerendsen, Inhomogeneous_NPTBerendsen):
        a = Atoms(atoms.numbers, atoms.positions, atoms.cell)
        v0 = a.get_volume()
        md = cls(a, PairCalc(), timestep=2.0, temperature=300.0, pressure=0.0, bulk_modulus=50.0)
        md.step()
        assert a.get_volume() > v0, cls.__name__


def test_thermostat_units():
    # dt / tau_t is a ratio of times; T = K_tr / (3 N k_B) is ASE's get_temperature for unconstrained atoms
    rng = np.random.default_rng(8)
    atoms = _crystal(rng)
    atoms.velocities = rng.normal(size=atoms.positions.shape) * 0.02
    md = NVTBerendsen(atoms, PairCalc(), timestep=2.0, temperature=300.0)
    assert abs(md.dt_over_taut - 0.01) < 1e-15 and abs(md.dt - 2.0 * FS) < 1e-15
    m = atoms.get_masses()[:, None]
    assert abs(md.temperature() - (m * atoms.velocities**2).sum() / (3 * len(atoms) * KB)) < 1e-9
