"""ms per DeviceMD step for nve / nvt / npt (per-axis and isotropic Berendsen) at 10,000 atoms (skin = 0: exact lists
rebuilt on the device every step) and at 64 / 288 atoms (skin 0.5: one CUDA-graph replay per step).  Every entry
carries the device name and its power limit.  Host clock around a synchronised window of >= 200 steps after warm-up.

    python tools/time_md_ensembles.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from chgnet_b200 import graphgen  # noqa: E402
from chgnet_b200.dynamics_device import DeviceMD  # noqa: E402
from chgnet_b200.model import CHGNet  # noqa: E402

ENSEMBLES = {
    "nve": dict(ensemble="nve"),
    "nvt": dict(ensemble="nvt", thermostat="Berendsen_inhomogeneous"),
    "npt_inhomogeneous": dict(ensemble="npt", thermostat="Berendsen_inhomogeneous", bulk_modulus=150.0),
    "npt_isotropic": dict(ensemble="npt", thermostat="npt_berendsen", bulk_modulus=150.0),
}
SIZES = {64: ((2, 2, 2), 0.5, 400), 288: ((3, 3, 4), 0.5, 400), 10000: ((10, 5, 25), 0.0, 200)}


def device_info() -> dict:
    idx = torch.cuda.current_device()
    info = {"device": torch.cuda.get_device_name(idx), "power_limit_w": None}
    try:  # a read-only query
        out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001  (no nvidia-smi: the name alone)
        pass
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--warmup", type=int, default=30)
    args = ap.parse_args()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    model = CHGNet.from_file(os.path.join(root, "tests", "golden", "chgnet_0.3.0_weights.npz"), version="0.3.0").to("cuda")
    info = device_info()
    rows = []
    for n_atoms, (reps, skin, steps) in SIZES.items():
        z, frac, lat = graphgen.limno2_structure(reps, 0.02, 77)
        assert len(z) == n_atoms, len(z)
        for name, kw in ENSEMBLES.items():
            md = DeviceMD(model, z, frac @ lat, lat, timestep=2.0, skin=skin, **kw)
            md.set_temperature(300.0, seed=1)
            md.run(args.warmup, log_every=0)
            torch.cuda.synchronize()
            b0, s0 = md.n_builds, md.n_strain_builds
            t0 = time.perf_counter()
            md.run(steps, log_every=0)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / steps
            row = {**info, "atoms": n_atoms, "ensemble": name, "skin": skin, "cuda_graph": md.use_cuda_graph, "steps": steps,
                   "ms_per_step": round(dt * 1e3, 4), "list_builds": md.n_builds - b0, "strain_builds": md.n_strain_builds - s0}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del md
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
