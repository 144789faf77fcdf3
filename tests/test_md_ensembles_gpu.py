"""-m gpu: the Berendsen NVT / NPT ensembles of DeviceMD (chgnet_b200/dynamics_device.py, csrc/md.cu) against the host
checkers of chgnet_b200/dynamics.py (ASE's NVTBerendsen / NPTBerendsen / Inhomogeneous_NPTBerendsen restated, one
CHGNetCalculator call per step, the reference's MolecularDynamics ensembles, dynamics.py:595-715), against themselves
(CUDA graph vs eager, skin vs exact lists, run vs run) and against loose physical expectations."""
import os

import numpy as np
import pytest
import torch

from chgnet_b200 import graphgen

pytestmark = pytest.mark.gpu

# (ensemble, thermostat) -> host checker
CASES = {
    "nvt": ("nvt", "Berendsen_inhomogeneous"),
    "npt_inhomogeneous": ("npt", "Berendsen_inhomogeneous"),
    "npt_isotropic": ("npt", "npt_berendsen"),
}


@pytest.fixture(scope="module")
def model():
    from chgnet_b200.model import CHGNet

    path = os.path.join(os.path.dirname(__file__), "golden", "chgnet_0.3.0_weights.npz")
    return CHGNet.from_file(path, version="0.3.0").to("cuda")


def _system(seed=4300, supercell=(2, 2, 1), shear=True, scale=1.0):
    z, frac, lat = graphgen.limno2_structure(supercell, 0.03, seed)
    lat = lat * scale
    if shear:  # triclinic: b and c lean over a
        lat = lat.copy()
        lat[1, 0] += 0.35
        lat[2, 0] -= 0.25
        lat[2, 1] += 0.2
    return z, frac @ lat, lat


def _host(case, model, atoms, **kw):
    from chgnet_b200.dynamics import CHGNetCalculator, Inhomogeneous_NPTBerendsen, NPTBerendsen, NVTBerendsen

    calc = CHGNetCalculator(model=model, on_isolated_atoms="ignore")
    cls = {"nvt": NVTBerendsen, "npt_inhomogeneous": Inhomogeneous_NPTBerendsen, "npt_isotropic": NPTBerendsen}[case]
    if case == "nvt":
        kw = {k: v for k, v in kw.items() if k in ("timestep", "temperature", "taut")}
    return cls(atoms, calc, **kw)


COUPLING = dict(timestep=2.0, temperature=450.0, pressure=1.0, taut=40.0, taup=100.0, bulk_modulus=100.0)


@pytest.mark.parametrize("case", list(CASES))
def test_device_trajectory_equals_the_host_checker(model, case):
    from chgnet_b200.dynamics import Atoms
    from chgnet_b200.dynamics_device import DeviceMD

    ens, th = CASES[case]
    z, pos, cell = _system()
    steps = 50
    atoms = Atoms(z, pos, cell)
    host = _host(case, model, atoms, **COUPLING)
    host.set_temperature(300.0, seed=7)
    v0 = atoms.velocities.copy()
    kw = dict(COUPLING, ensemble=ens, thermostat=th, velocities=v0)
    if ens == "nvt":
        kw.pop("bulk_modulus")
    exact = DeviceMD(model, z, pos, cell, skin=0.0, **kw)
    graph = DeviceMD(model, z, pos, cell, skin=0.5, use_cuda_graph=True, **kw)
    assert abs(exact.kinetic_energy - host.kinetic_energy()) < 1e-9  # correct before the first step
    hlog = host.run(steps)
    logs = [exact.run(steps), graph.run(steps)]
    for md, log in zip((exact, graph), logs):
        dx = np.abs(md.positions() - atoms.positions).max()
        dc = np.abs(md.cell() - atoms.cell).max()
        print(f"{case} skin {md.skin}: 50 steps |x_dev - x_host| = {dx:.2e} A, |L_dev - L_host| = {dc:.2e} A, "
              f"builds {md.n_builds} (strain {md.n_strain_builds}), V {cell[0] @ np.cross(cell[1], cell[2]):.3f} -> {md.volume:.3f}")
        assert dx < 1e-4 and dc < 1e-5, (dx, dc)
        for h, d in zip(hlog[9::10], log[9::10]):
            assert abs(h["e_pot"] - d["e_pot"]) < 1e-3 and abs(h["e_kin"] - d["e_kin"]) < 1e-3, (h, d)
            if "volume" in h:
                assert abs(h["volume"] - d["volume"]) < 1e-3 and abs(h["pressure"] - d["pressure"]) < 1e-2, (h, d)
    assert graph.n_builds < 12
    if ens == "npt":
        assert np.abs(atoms.cell - cell).max() > 1e-3  # the barostat did move the cell


@pytest.mark.parametrize("case", list(CASES))
def test_cuda_graph_step_equals_the_eager_step(model, case):
    from chgnet_b200.dynamics_device import DeviceMD

    ens, th = CASES[case]
    z, pos, cell = _system(4301)
    kw = dict(timestep=1.0, ensemble=ens, thermostat=th, taut=20.0, taup=50.0, bulk_modulus=100.0, temperature=600.0)
    a = DeviceMD(model, z, pos, cell, skin=0.6, use_cuda_graph=True, **kw)
    b = DeviceMD(model, z, pos, cell, skin=0.6, use_cuda_graph=False, **kw)
    for md in (a, b):
        md.set_temperature(500.0, seed=3)
    a.run(12, log_every=0)
    b.run(12, log_every=0)
    assert a.n_captures >= 1
    assert np.abs(a.positions() - b.positions()).max() < 1e-9
    assert np.abs(a.cell() - b.cell()).max() < 1e-12
    assert abs(a.potential_energy - b.potential_energy) < 1e-7


def _launch_step(lib, st, t, flags, dt, with_kick=True):
    n = t["x"].shape[0]
    assert lib.chg_md_cell_step(t["par"].data_ptr(), t["cs"].data_ptr(), t["k"].data_ptr(), n, t["vir"].data_ptr(), t["lat"].data_ptr(),
                                flags, st) == 0
    assert lib.chg_md_kick_drift_cell(t["x"].data_ptr(), t["v"].data_ptr(), t["f"].data_ptr(), t["im"].data_ptr(), n, dt,
                                      t["cs"].data_ptr(), t["mom"].data_ptr(), t["f64"].data_ptr(), t["f32"].data_ptr(),
                                      t["sref"].data_ptr(), flags, st) == 0
    assert lib.chg_md_kick_partials(t["v"].data_ptr(), t["f"].data_ptr(), t["im"].data_ptr(), n, dt, t["k"].data_ptr(), st) == 0


@pytest.mark.parametrize("flags", [1, 1 | 8, 1 | 2 | 8, 1 | 4 | 8, 1 | 4])
def test_integrator_kernels_are_deterministic_and_follow_the_step(flags):
    """The chg_md_* kernels alone (fixed forces and virial, 5,000 atoms = 20 blocks of partials): two runs are bit for bit
    the same (no atomics feed the trajectory), and every quantity follows the numpy restatement of the step."""
    from chgnet_b200.dynamics import ATOMIC_MASSES, FS, GPA, KB, berendsen_lambda
    from chgnet_b200.dynamics_device import _lib

    lib, dev = _lib(), torch.device("cuda")
    rng = np.random.default_rng(flags)
    n, dt, steps = 5000, 2.0 * FS, 6
    lat = np.array([[38.0, 0.0, 0.0], [3.1, 35.0, 0.0], [-2.2, 1.7, 41.0]])
    m = ATOMIC_MASSES[rng.integers(1, 80, n)]
    x0 = rng.random((n, 3)) @ lat
    v0 = rng.normal(size=(n, 3)) * np.sqrt(KB * 700.0 / m)[:, None] + 0.002
    f = rng.normal(size=(n, 3)) * 0.7
    f -= f.mean(axis=0)  # Newton's third law: the kicks add no momentum
    vir = rng.normal(size=(3, 3)) * 5.0
    vir = vir + vir.T - 20.0 * np.eye(3)  # compressive
    mask = np.array([1.0, 0.0, 1.0])
    par = np.array([450.0, 1.5 * GPA, 0.2, dt / (30.0 * FS) / (80.0 * GPA) / 3.0, *mask, KB])
    inv = np.linalg.inv(lat)

    def fresh():
        cs = np.zeros(64)
        cs[0:9], cs[9:18], cs[18:27], cs[27:36], cs[36:45], cs[45] = lat.ravel(), inv.ravel(), inv.ravel(), lat.ravel(), inv.ravel(), abs(np.linalg.det(lat))
        d = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        nblk = int(lib.chg_md_partial_blocks(n))
        t = {"x": d(x0), "v": d(v0), "f": d(f), "im": d(1.0 / m), "vir": d(vir.ravel()), "par": d(par), "cs": d(cs),
             "k": torch.zeros(nblk, 4, dtype=torch.float64, device=dev), "mom": torch.zeros(nblk, 3, dtype=torch.float64, device=dev),
             "f64": torch.empty(n, 3, dtype=torch.float64, device=dev), "f32": torch.empty(n, 3, dtype=torch.float32, device=dev),
             "lat": torch.zeros(1, 9, dtype=torch.float32, device=dev), "sref": d(x0 @ inv)}
        st = torch.cuda.current_stream().cuda_stream
        assert lib.chg_md_kick_partials(t["v"].data_ptr(), None, t["im"].data_ptr(), n, 0.0, t["k"].data_ptr(), st) == 0
        for _ in range(steps):
            _launch_step(lib, st, t, flags, dt)
        torch.cuda.synchronize()
        return {k: v.cpu().numpy() for k, v in t.items()}

    a, b = fresh(), fresh()
    for key in ("x", "v", "cs", "k", "f64", "f32", "lat"):
        assert np.array_equal(a[key], b[key]), key

    # numpy restatement of the same six steps
    x, v, L = x0.copy(), v0.copy(), lat.copy()
    for _ in range(steps):
        k = (m[:, None] * v * v).sum(axis=0)
        lam = berendsen_lambda(k.sum() / (3 * n * KB), par[0], par[2])
        vol = abs(np.linalg.det(L))
        mu = np.ones(3)
        if flags & 6:
            p = (lam * lam * k - np.diag(vir)) / vol
            mu = 1.0 - par[3] * (par[1] - p) * mask if flags & 4 else np.full(3, 1.0 - par[3] * (par[1] - p.sum() / 3.0))
        l_new = mu[:, None] * L
        x = (x @ np.linalg.inv(L)) @ l_new
        L = l_new
        v = lam * v + 0.5 * dt * f / m[:, None]
        if flags & 8:
            v = v - (m[:, None] * v).sum(axis=0) / n / m[:, None]
        x = x + dt * v
        v = v + 0.5 * dt * f / m[:, None]
    s = x @ np.linalg.inv(L)
    assert np.abs(a["x"] - x).max() < 1e-9 and np.abs(a["v"] - v).max() < 1e-12
    assert np.abs(a["cs"][0:9].reshape(3, 3) - L).max() < 1e-12
    assert np.abs(a["cs"][9:18].reshape(3, 3) - np.linalg.inv(L)).max() < 1e-15
    assert abs(a["cs"][45] - abs(np.linalg.det(L))) < 1e-8 * abs(np.linalg.det(L))
    assert np.abs(a["f64"] - s).max() < 1e-12 and np.array_equal(a["f32"], a["f64"].astype(np.float32))
    assert np.abs(a["k"].sum(axis=0)[:3] - (m[:, None] * v * v).sum(axis=0)).max() < 1e-9 * (m[:, None] * v * v).sum()
    d2 = ((((s - x0 @ inv) @ lat) ** 2).sum(axis=1)).max()
    eps = np.linalg.norm(inv @ L - np.eye(3))
    assert abs(a["cs"][52] - d2) < 1e-9 * max(d2, 1e-12) and abs(a["cs"][53] - eps) < 1e-12
    if flags & 6:
        assert eps > 1e-4  # the barostat moved the cell
    if flags & 8:
        assert np.abs((m[:, None] * a["v"]).sum(axis=0)).max() < 1e-9
    if flags & 4:
        assert np.array_equal(a["cs"][3:6], lat[1])  # masked lattice vector untouched


@pytest.mark.parametrize("case", list(CASES))
def test_repeated_runs_agree(model, case):
    # chg_forward adds some force contributions with floating-point atomics, so two runs of the same trajectory agree to
    # rounding rather than bit for bit; the integrator's own sums are ordered (test above)
    from chgnet_b200.dynamics_device import DeviceMD

    ens, th = CASES[case]
    z, pos, cell = _system(4302)
    out = []
    for _ in range(2):
        md = DeviceMD(model, z, pos, cell, skin=0.5, ensemble=ens, thermostat=th, taup=50.0, bulk_modulus=100.0)
        md.set_temperature(400.0, seed=5)
        md.run(20, log_every=0)
        out.append((md.positions(), md.v.cpu().numpy(), md.cell()))
    for a, b in zip(*out):
        assert np.abs(a - b).max() < 1e-9


def test_skin_survives_a_deforming_cell(model):
    from chgnet_b200.dynamics_device import DeviceMD

    z, pos, cell = _system(4303, scale=0.96)
    kw = dict(timestep=2.0, ensemble="npt", thermostat="Berendsen_inhomogeneous", pressure=0.0, taup=20.0, bulk_modulus=100.0)
    skin = DeviceMD(model, z, pos, cell, skin=0.5, **kw)
    exact = DeviceMD(model, z, pos, cell, skin=0.0, **kw)
    for md in (skin, exact):
        md.set_temperature(300.0, seed=9)
    skin.run(40, log_every=0)
    exact.run(40, log_every=0)
    dx = np.abs(skin.positions() - exact.positions()).max()
    print(f"compressed cell, taup 20 fs: {skin.n_builds} builds ({skin.n_strain_builds} from the strain), "
          f"V {abs(np.linalg.det(cell)):.2f} -> {skin.volume:.2f}, |x_skin - x_exact| = {dx:.2e} A")
    assert skin.n_strain_builds >= 1
    assert skin.volume > abs(np.linalg.det(cell)) * 1.02
    assert dx < 1e-4 and np.abs(skin.cell() - exact.cell()).max() < 1e-5


def test_set_target_keeps_the_captured_step(model):
    from chgnet_b200.dynamics_device import DeviceMD

    z, pos, cell = _system(4304)
    kw = dict(timestep=2.0, ensemble="npt", thermostat="npt_berendsen", taut=20.0, taup=100.0, bulk_modulus=100.0)
    a = DeviceMD(model, z, pos, cell, skin=1.0, use_cuda_graph=True, **kw)
    b = DeviceMD(model, z, pos, cell, skin=1.0, use_cuda_graph=False, **kw)
    for md in (a, b):
        md.set_temperature(300.0, seed=1)
        md.run(10, log_every=0)
    captures, builds, graph = a.n_captures, a.n_builds, a.graph
    for md in (a, b):
        md.set_target(temperature=900.0, pressure=2.0)
    assert graph is not None and a.graph is graph
    for md in (a, b):
        md.run(15, log_every=0)
    assert a.n_captures - captures <= a.n_builds - builds  # only a list rebuild recaptures
    assert np.abs(a.positions() - b.positions()).max() < 1e-9 and np.abs(a.cell() - b.cell()).max() < 1e-12
    assert a.temperature() > 400.0


def test_nvt_reaches_the_target_temperature(model):
    from chgnet_b200.dynamics_device import DeviceMD

    z, pos, cell = _system(4305, supercell=(2, 2, 2), shear=False)
    md = DeviceMD(model, z, pos, cell, timestep=2.0, skin=0.5, ensemble="nvt", temperature=600.0, taut=10.0)
    md.set_temperature(300.0, seed=2)
    t0 = md.temperature()
    log = md.run(300)
    tail = np.mean([e["temperature"] for e in log[200:]])
    print(f"NVT taut = 5 dt: T {t0:.0f} K -> mean {tail:.0f} K over the last 100 steps (target 600 K)")
    assert abs(t0 - 300.0) < 60.0
    assert abs(tail - 600.0) < 60.0


def test_npt_relaxes_a_compressed_cell(model):
    from chgnet_b200.dynamics_device import DeviceMD

    z, pos, cell = _system(4306, shear=False, scale=0.98)
    md = DeviceMD(model, z, pos, cell, timestep=2.0, skin=0.5, ensemble="npt", thermostat="Berendsen_inhomogeneous",
                  taup=50.0, bulk_modulus=100.0)
    p_target = 1.01325e-4
    v0, p0 = md.volume, md.pressure()
    log = md.run(20)
    print(f"NPT from a 2 % compressed cell: V {v0:.2f} -> {log[-1]['volume']:.2f} A^3, P {p0:.2f} -> {log[-1]['pressure']:.2f} GPa")
    assert p0 > 1.0
    assert log[-1]["volume"] > v0
    assert abs(log[-1]["pressure"] - p_target) < abs(p0 - p_target)


def test_argument_errors_and_the_unchanged_nve_path(model):
    from chgnet_b200.dynamics_device import DeviceMD

    z, pos, cell = _system(4307, shear=False)
    with pytest.raises(ValueError, match="Ensemble"):
        DeviceMD(model, z, pos, cell, ensemble="nph")
    with pytest.raises(ValueError, match="Thermostat not supported"):
        DeviceMD(model, z, pos, cell, ensemble="nvt", thermostat="Andersen")
    with pytest.raises(NotImplementedError, match="Nose-Hoover"):
        DeviceMD(model, z, pos, cell, ensemble="nvt", thermostat="Nose-Hoover")
    with pytest.raises(ValueError, match="bulk_modulus"):
        DeviceMD(model, z, pos, cell, ensemble="npt")
    plain = DeviceMD(model, z, pos, cell, skin=0.5)
    nve = DeviceMD(model, z, pos, cell, skin=0.5, ensemble="nve", thermostat="Berendsen", temperature=900.0, pressure=3.0,
                   taut=5.0, taup=5.0, bulk_modulus=1.0, fix_com=False, mask=(0, 0, 1))
    for md in (plain, nve):
        md.set_temperature(300.0, seed=4)
        assert abs(md.temperature() - 300.0) < 100.0  # known before the first step
    plain.run(15, log_every=0)
    nve.run(15, log_every=0)
    assert plain.n_builds == nve.n_builds and plain.n_captures == nve.n_captures
    assert np.abs(plain.positions() - nve.positions()).max() < 1e-9  # chg_forward's atomics: equal to rounding
    assert np.array_equal(plain.cell(), cell) and plain.volume == pytest.approx(abs(np.linalg.det(cell)))
    with pytest.raises(ValueError, match="set_target"):
        plain.set_target(temperature=10.0)
    torch.cuda.synchronize()
