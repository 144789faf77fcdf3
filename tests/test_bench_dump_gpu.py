"""-m gpu: bench.py --dump-outputs writes what the timed path computed in its last step, the same from run to run,
and for the c1 workload (LiMnO2) the same as the fp64 oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from chgnet_b200 import graphgen
from oracle import chgnet_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                          "--dump-outputs", str(out_dir), *args], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_inference_dump_is_repeatable_and_matches_oracle(tmp_path, weights030):
    a = _bench(tmp_path / "a", "--workload", "c1")
    b = _bench(tmp_path / "b", "--workload", "c1")
    assert sorted(a) == ["energy", "force", "stress"]
    assert a["energy"].shape == (1,) and a["energy"].dtype == np.float64
    assert a["force"].shape == (8, 3) and a["force"].dtype == np.float32
    assert a["stress"].shape == (1, 3, 3) and a["stress"].dtype == np.float32
    for k in a:
        np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6, err_msg=k)

    z, frac, lat = graphgen.limno2_structure()
    g = graphgen.make_crystal_graph(z, frac, lat, graph_id="mp-18767")
    ref = orc.predict_graph(weights030, g, "efs", dtype=torch.float64)
    # the dumped energy is the network's total, before the AtomRef composition term; the oracle's `e` is per atom with it
    wref = np.asarray(weights030["composition_model.fc.weight"], np.float64)[0]
    n = len(z)
    assert abs(float(a["energy"][0]) - (float(ref["e"]) * n - wref[np.asarray(z) - 1].sum())) < 1e-4 * n
    assert np.max(np.abs(a["force"] - ref["f"])) < 1e-3
    assert np.max(np.abs(a["stress"][0] - ref["s"])) < 1e-3


@pytest.mark.gpu
def test_training_dump(tmp_path):
    d = _bench(tmp_path, "--workload", "c5")
    assert {"loss", "grad", "params"} <= set(d)
    assert d["grad"].ndim == 1 and d["grad"].shape == d["params"].shape and d["params"].dtype == np.float32
    assert d["loss"].shape == () and float(d["loss"]) > 0
    for k, v in d.items():
        assert np.all(np.isfinite(v)), k
