"""-m gpu: end-to-end parity of chgnet_b200.CHGNet (CUDA kernels through the C ABI)
against the committed golden vectors of the live reference, the fp64 oracle, and the
invariants the reference's own tests pin (reference tests/test_model.py:60-219)."""
import os

import numpy as np
import pytest
import torch

from chgnet_b200 import graphgen

pytestmark = pytest.mark.gpu

# north-star tolerances (BASELINE.json): 1e-4 eV/atom, 1e-3 eV/A, 1e-3 GPa (and 1e-3 muB)
TOL = {"e": 1e-4, "f": 1e-3, "s": 1e-3, "m": 1e-3}


@pytest.fixture(scope="module")
def model():
    from chgnet_b200.model import CHGNet

    path = os.path.join(os.path.dirname(__file__), "golden", "chgnet_0.3.0_weights.npz")
    return CHGNet.from_file(path, version="0.3.0").to("cuda")


def _maxabs(a, b):
    return float(np.max(np.abs(np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64))))


def test_limno2_known_answers(model, limno2_graph, golden):
    out = model.predict_graph(limno2_graph, return_site_energies=True, return_atom_feas=True,
                              return_crystal_feas=True)
    assert sorted(out) == ["atom_fea", "crystal_fea", *"efms", "site_energies"]
    # published known answers (reference tests/test_model.py:68-119)
    assert out["e"] == pytest.approx(-7.36769, rel=1e-4, abs=1e-4)
    assert out["e"].shape == () and out["f"].shape == (8, 3) and out["s"].shape == (3, 3)
    assert out["crystal_fea"].mean() == pytest.approx(0.26999, rel=1e-4, abs=1e-4)
    assert out["atom_fea"].mean() == pytest.approx(-0.09668, rel=1e-4, abs=1e-4)
    assert out["crystal_fea"].shape == (64,) and out["atom_fea"].shape == (8, 64)
    assert np.sum(out["site_energies"]) / 8 == pytest.approx(out["e"], rel=1e-4, abs=1e-6)
    # live-reference fp32 outputs and fp64 truth, at the north-star tolerances
    for tag in ("ref32", "oracle64"):
        for k, tol in TOL.items():
            err = _maxabs(out[k], golden[f"limno2.{tag}.{k}"])
            assert err < tol, (tag, k, err)
        assert _maxabs(out["site_energies"], golden[f"limno2.{tag}.site_energies"]) < 1e-4
    print({k: f"{_maxabs(out[k], golden[f'limno2.oracle64.{k}']):.2e}" for k in TOL})


@pytest.mark.parametrize("ws_min_rows", [0, 4096], ids=["tcgen05-ws-forced", "defaults-ffma"])
def test_limno2_parity_for_every_implementation(model, limno2_graph, golden, ws_min_rows):
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    K.set_option("ws_min_rows", ws_min_rows)  # 8-atom cell: 0 forces the warp-specialised tcgen05 kernels
    try:
        out = model.predict_graph(limno2_graph)
        for k, tol in TOL.items():
            assert _maxabs(out[k], golden[f"limno2.oracle64.{k}"]) < tol, k
    finally:
        K.set_option("ws_min_rows", 4096)


def test_random_batch_vs_reference_golden(model, golden):
    graphs = graphgen.random_graphs(4, 12, 20, 7000)
    preds = model.predict_graph(graphs, task="efsm", batch_size=4)
    assert isinstance(preds, list) and len(preds) == 4
    for i, p in enumerate(preds):
        for tag in ("ref32", "oracle64"):
            for k, tol in TOL.items():
                assert _maxabs(p[k], golden[f"rand4.{i}.{tag}.{k}"]) < tol, (i, tag, k)


def test_batched_equals_single_and_batch_size(model):
    graphs = graphgen.random_graphs(5, 8, 14, 7100)
    together = model.predict_graph(graphs, batch_size=16)
    chunked = model.predict_graph(graphs, batch_size=2)
    for g, a, b in zip(graphs, together, chunked):
        single = model.predict_graph(g)
        for k, tol in TOL.items():
            assert _maxabs(a[k], single[k]) < tol * 0.1 and _maxabs(a[k], b[k]) < tol * 0.1


def test_against_fp64_oracle_on_larger_batch(model, weights030):
    from oracle import chgnet_oracle as orc

    graphs = graphgen.random_graphs(6, 24, 40, 7200)
    preds = model.predict_graph(graphs, task="efsm", batch_size=6)
    ref = orc.predict_graph(weights030, graphs, "efsm", batch_size=6, dtype=torch.float64)
    worst = {k: max(_maxabs(p[k], r[k]) for p, r in zip(preds, ref)) for k in TOL}
    print("max |cuda - oracle64|:", {k: f"{v:.2e}" for k, v in worst.items()})
    for k, tol in TOL.items():
        assert worst[k] < tol, (k, worst[k])


def test_rotation_and_supercell_invariance(model):
    """reference tests/test_model.py:122-191"""
    z, frac, lat = graphgen.random_structure(10, 7300)
    base = model.predict_structure((z, frac, lat))
    th = np.deg2rad(30.0)
    axis = np.array([-2.0, 3.0, 1.0]) / np.linalg.norm([-2.0, 3.0, 1.0])
    Kx = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    Rm = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
    rot = model.predict_structure((z, frac, lat @ Rm.T))
    assert rot["e"] == pytest.approx(base["e"], abs=1e-4)
    assert _maxabs(rot["f"], base["f"] @ Rm.T) < 1e-3
    assert _maxabs(rot["s"], Rm @ base["s"] @ Rm.T) < 1e-3
    assert _maxabs(rot["m"], base["m"]) < 1e-3
    # 2x1x1 supercell: same energy per atom, forces tiled
    frac2 = np.concatenate([frac / [2, 1, 1], frac / [2, 1, 1] + [0.5, 0, 0]])
    sup = model.predict_structure((np.tile(z, 2), frac2, lat * np.array([[2], [1], [1]])))
    assert sup["e"] == pytest.approx(base["e"], abs=1e-4)
    assert _maxabs(sup["f"], np.tile(base["f"], (2, 1))) < 1e-3
    assert _maxabs(sup["s"], base["s"]) < 1e-3


def test_tasks_keys_and_errors(model, limno2_graph):
    out = model([limno2_graph])
    assert list(out) == ["atoms_per_graph", "e"]  # reference tests/test_model.py:47
    assert out["atoms_per_graph"].shape == (1,) and out["e"] < 0
    for task, keys in (("e", "e"), ("ef", "ef"), ("em", "em"), ("efs", "efs"), ("efsm", "efms")):
        assert sorted(model.predict_graph(limno2_graph, task=task)) == sorted(keys)
    with pytest.raises(ValueError, match="Invalid task='abc'"):
        model.predict_graph(limno2_graph, task="abc")
    with pytest.raises(TypeError, match="must be CrystalGraph or list of CrystalGraphs"):
        model.predict_graph(3)


def test_isolated_atoms_and_empty_bond_graph(model, weights030):
    from oracle import chgnet_oracle as orc

    g_far = graphgen.make_crystal_graph([3, 8], np.array([[0.0, 0, 0], [0.5, 0.5, 0.5]]), np.eye(3) * 5.5)
    g_iso = graphgen.make_crystal_graph([1, 1], np.array([[0.0, 0, 0], [0.5, 0.5, 0.5]]), np.eye(3) * 20.0)
    assert len(g_far.bond_graph) == 0 and len(g_iso.atom_graph) == 0
    for graphs in ([g_far], [g_iso], [g_iso, g_far], graphgen.random_graphs(1, 9, 9, 7400) + [g_iso]):
        preds = model.predict_graph(graphs, task="efsm")
        ref = orc.predict_graph(weights030, graphs, "efsm", dtype=torch.float64)
        for p, r in zip(preds, ref):
            for k, tol in TOL.items():
                assert _maxabs(p[k], r[k]) < tol
    g10 = graphgen.make_crystal_graph([1, 1], np.array([[0.0, 0, 0], [0.5, 0.5, 0.5]]), np.eye(3) * 10.0)
    e10, e20 = model.predict_graph(g10)["e"], model.predict_graph(g_iso)["e"]
    assert e10 == pytest.approx(e20, rel=1e-5, abs=1e-5)  # reference tests/test_model.py:210-219


def test_state_dict_round_trip(model):
    from chgnet_b200.model import CHGNet

    dct = model.as_dict()
    assert {*dct} == {"model_args", "state_dict"} and len(dct["state_dict"]) == 136
    clone = CHGNet.from_dict(dct).to("cuda")
    assert clone.n_params == 412525
    g = graphgen.random_graphs(1, 8, 8, 7500)[0]
    a, b = model.predict_graph(g), clone.predict_graph(g)
    assert all(np.array_equal(a[k], b[k]) for k in "efsm")


def test_large_cell_properties(model):
    """Size-independent checks at a config-4-like size (LiMnO2 6x4x3 = 576 atoms):
    net force ~ 0 (translation invariance), stress symmetric, results reproducible."""
    z, frac, lat = graphgen.limno2_structure((6, 4, 3), 0.02, 4000)
    g = graphgen.make_crystal_graph(z, frac, lat)
    a = model.predict_graph(g)
    b = model.predict_graph(g)
    assert np.abs(a["f"].sum(axis=0)).max() < 1e-3
    assert _maxabs(a["s"], a["s"].T) < 1e-3
    assert np.array_equal(a["e"], b["e"]) and _maxabs(a["f"], b["f"]) < 1e-5


def test_v020_shaped_architecture_end_to_end(weights030):
    """Constructor + pack_weights + kernels for the 0.2.0 architecture (9 radial / 9 angular functions,
    no LayerNorm, mlp_out bias, two readout hidden layers, cutoff_coeff 5, 5 A atom-graph cutoff) with
    random weights, against the oracle fed the SAME state_dict."""
    from chgnet_b200.model import CHGNet
    from oracle import chgnet_oracle as orc

    torch.manual_seed(3)
    m = CHGNet(num_radial=9, num_angular=9, gMLP_norm=None, readout_norm=None, mlp_hidden_dims=[64, 64],
               cutoff_coeff=5, atom_graph_cutoff=5, mlp_out_bias=True, composition_model="MPtrj").to("cuda")
    sd = m.state_dict()
    assert len(sd) == 99 and m.n_params == 400438  # reference tests/test_model.py:236-310 (0.2.0 counts)
    assert "atom_conv_layers.0.mlp_out.layers.1.bias" in sd and "readout_norm.weight" not in sd
    w = {k: v.detach().cpu().numpy() for k, v in sd.items()}
    args = dict(num_radial=9, num_angular=9, gMLP_norm=None, readout_norm=None, mlp_out_bias=True, cutoff_coeff=5,
                atom_graph_cutoff=5.0)
    graphs = graphgen.random_graphs(3, 8, 14, 7600, atom_graph_cutoff=5.0)
    preds = m.predict_graph(graphs, task="efsm", batch_size=3)
    ref = orc.predict_graph(w, graphs, "efsm", batch_size=3, dtype=torch.float64, args=args)
    for p, r in zip(preds, ref):
        for k, tol in TOL.items():
            assert _maxabs(p[k], r[k]) < tol * 5, (k, _maxabs(p[k], r[k]))  # untrained weights: larger magnitudes


def test_native_forward_equals_python_schedule(model, monkeypatch):
    """chg_forward (one C call, native schedule + workspace) == engine.py calling the same kernels one by one."""
    from chgnet_b200.batch import build_batch

    graphs = graphgen.random_graphs(5, 10, 24, 7700)
    kw = dict(task="efsm", return_site_energies=True, return_atom_feas=True, return_crystal_feas=True, batch_size=5)
    nat = model.predict_graph(graphs, **kw)
    calls = model._get_native().calls
    assert calls >= 1
    monkeypatch.setenv("CHGNET_B200_ENGINE", "python")
    py = model.predict_graph(graphs, **kw)
    assert model._get_native().calls == calls  # the Python schedule really ran
    monkeypatch.delenv("CHGNET_B200_ENGINE")
    for a, b in zip(nat, py):
        assert set(a) == set(b)
        for k in a:
            # same kernels, same order: identical up to the order of the fp64 atomics in force / virial
            assert _maxabs(a[k], b[k]) <= 1e-6 * max(1.0, float(np.abs(b[k]).max())), k
    # energy-only call, then a larger batch: the workspace grows and is reused
    e_only = model.predict_graph(graphs[:2], task="e", batch_size=2)
    assert _maxabs(e_only[0]["e"], nat[0]["e"]) < 1e-6
    big = model.predict_graph(graphgen.random_graphs(12, 20, 30, 7800), task="efs", batch_size=12)
    assert len(big) == 12 and np.isfinite(big[3]["f"]).all()
    # a workspace that is too small is an error, not a crash
    import ctypes

    from chgnet_b200 import native

    n = model._get_native()
    b = build_batch(graphs, model.device)
    res = {"energy": torch.empty(5, dtype=torch.float64, device="cuda"), "e_ref": torch.empty(5, dtype=torch.float64, device="cuda"),
           "site_e": torch.empty(b.n_atoms, device="cuda")}
    outs = native.Outputs(**{k: v.data_ptr() for k, v in res.items()})
    bs = native.batch_struct(b)
    small = torch.empty(1 << 16, dtype=torch.uint8, device="cuda")
    base = (small.data_ptr() + 255) // 256 * 256
    rc = n.lib.chg_forward(ctypes.byref(n.hps), n.weights.data_ptr(), ctypes.byref(bs), ctypes.byref(outs), base, 1 << 15,
                           torch.cuda.current_stream().cuda_stream)
    assert rc != 0 and b"workspace too small" in n.lib.chg_last_error()


def test_static_evaluator_replays_one_cuda_graph():
    """CHGNet.static_evaluator: fixed topology, coordinates updated in place, chg_forward replayed as a CUDA graph
    (NativeForward.replay).  Same numbers as predict_graph on the re-built graph of the displaced structure, call after
    call (eager -> capture -> replays), for a single graph and for a list."""
    from chgnet_b200.model import CHGNet

    gold = os.path.join(os.path.dirname(__file__), "golden", "chgnet_0.3.0_weights.npz")
    model = CHGNet.from_file(gold, version="0.3.0").to("cuda")
    rng = np.random.default_rng(5)
    structs = [graphgen.random_structure(n, 4100 + n) for n in (12, 17)]
    graphs = [graphgen.make_crystal_graph(*s) for s in structs]
    ev = model.static_evaluator(graphs, task="efsm")
    base = model.predict_graph(graphs, task="efsm", batch_size=2)
    calls_before = model._get_native().calls
    for it in range(5):
        new = [(z, f + (0.0015 * rng.standard_normal(f.shape) if it else 0.0), lat) for z, f, lat in structs]
        ev.update(frac=np.concatenate([f for _, f, _ in new]))
        got = ev()
        want = model.predict_graph([graphgen.make_crystal_graph(*s) for s in new], task="efsm", batch_size=2) if it else base
        for a, b in zip(got, want):
            assert set(a) == set(b)
            for k in b:
                assert np.abs(np.asarray(a[k], np.float64) - np.asarray(b[k], np.float64)).max() < 3e-5, (it, k)
    native = model._get_native()
    assert len(native._graphs) == 1 and native.calls > calls_before
    one = model.static_evaluator(graphs[0], task="ef")
    r = [one() for _ in range(3)]
    assert set(r[0]) == {"e", "f"} and np.allclose(r[0]["f"], r[2]["f"]) and np.allclose(r[0]["f"], base[0]["f"], atol=1e-6)
