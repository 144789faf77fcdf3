#!/usr/bin/env python
"""bench.py — throughput of the CHGNet hot path (E + F + sigma) on B200.

Contract (see task statement): ``python bench.py --gpus N --steps K --warmup W`` prints ONE
JSON line.  A "step" is one pass of the hot path (forward + the force/stress reverse pass)
over one batch of synthetic CrystalGraphs.

Workloads (SURVEY.md §8d, BASELINE.json `configs`):
  c3  (default) batch = 256 random cells, 20..40 atoms, cutoffs 6 A / 3 A          [configs[2]]
      the config the 1 -> 8 GPU curve is quoted on and the largest batched single-GPU one
  c2  batch = 64 random periodic cells, 40..60 atoms                               [configs[1]]
  c4  one 10,000-atom LiMnO2 supercell (10x5x25), sigma = 0.02 A displacements      [configs[3]]
      (also attached to every c2 / c3 line as the extra key "c4": the north-star's 10k-atom targets)
  c1  the 8-atom LiMnO2 cell                                                       [configs[0]]
  c5  fine-tuning step, batch = 128 (forward, CombinedLoss, double backward, all-reduce, Adam) [configs[4]]
      (at N > 1 a few c5 steps also run after the inference legs -> extra key "collective")

value      structures/s of the kernel path, batch descriptor already resident in HBM
e2e        the same through ``CHGNet.predict_graph`` from host CrystalGraphs (host packing,
           H2D, CSR build, kernels, D2H numpy) — the user-facing call
roofline   AtomConv scatter-reduce kernel (chg_segment_sum over center-sorted messages),
           timed alone with CUDA events at this workload's size, L2 flushed between launches
cpu_baseline / --impl reference
           the oracle port of the reference's torch CPU path (oracle/chgnet_oracle.py) on
           the host cores, on a bounded sample of the same workload

Multi-GPU: one process per GPU (torchrun).  The global batch (N x the workload's batch) is assigned to
ranks by `partition_graphs` (greedy LPT on edges + 2.5 x angles, chgnet_b200/batch.py); no device-path
collective for inference; time = max over ranks; weak scaling (per-GPU work fixed as N grows).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WEIGHTS = os.path.join(ROOT, "tests", "golden", "chgnet_0.3.0_weights.npz")
L2_FLUSH_BYTES = 256 << 20


def make_workload(name: str, rank: int, backend: str = "native"):
    """The workload's CrystalGraphs (deterministic; `rank` shifts the seeds).  backend="numpy" builds them
    without the kernel library (the reference arm must not map the product's .so)."""
    from chgnet_b200 import graphgen

    kw = {"backend": backend}
    if name == "c1":
        z, frac, lat = graphgen.limno2_structure()
        return [graphgen.make_crystal_graph(z, frac, lat, graph_id="mp-18767", **kw)], "LiMnO2 mp-18767, 8 atoms"
    if name == "c2":
        return graphgen.random_graphs(64, 40, 60, 1000 + 100 * rank, **kw), "batch=64 random periodic cells, 40..60 atoms, rho=0.10/A^3, cutoffs 6/3 A"
    if name == "c3":
        return graphgen.random_graphs(256, 20, 40, 2000 + 1000 * rank, **kw), "batch=256 random periodic cells, 20..40 atoms, rho=0.10/A^3, cutoffs 6/3 A"
    if name == "c4":
        z, frac, lat = graphgen.limno2_structure((10, 5, 25), 0.02, 4000 + rank)
        return [graphgen.make_crystal_graph(z, frac, lat, graph_id="LiMnO2-10x5x25", **kw)], "LiMnO2 10x5x25 supercell, 10,000 atoms, sigma=0.02 A"
    if name == "c5":
        return graphgen.random_graphs(128, 20, 40, 5000 + 1000 * rank, **kw), "fine-tune batch=128 random periodic cells, 20..40 atoms, rho=0.10/A^3, cutoffs 6/3 A; targets 'efsm' (MSE, ratios 1/1/0.1/0.1), Adam lr 1e-3"
    raise SystemExit(f"unknown workload {name}")


L2_NOTE = "256 MiB buffer written, then 256 MiB read (clean lines), between timed iterations"


def bench_config(workload: str, desc: str, per_job: dict, world: int, task: str = "efs") -> dict:
    """The `config` object, IDENTICAL in the product arm and in the reference arm (the driver compares them):
    the workload, the task, the whole-job sizes, the weights and how the L2 is treated between timed steps."""
    return {"workload": f"{workload}: {desc}", "task": task, "whole_job": per_job, "weights": "CHGNet 0.3.0",
            "l2": L2_NOTE, "parallelism": f"graph-sharded x{world} (LPT partition of the global batch), no inference collective"}


def sharded_workload(name: str, rank: int, world: int, backend: str = "native"):
    """(my graphs, description, whole-job counts).  N > 1: the global batch = the N per-rank batches of
    `make_workload`; every rank builds it, costs it, and keeps the share `partition_graphs` (greedy LPT)
    assigns to it - the partitioner of chgnet_b200/parallel.py::predict_sharded."""
    from chgnet_b200.batch import graph_cost, partition_graphs

    if world == 1 or name in ("c1", "c4"):  # a single structure does not shard: replicas (DESIGN.md §7)
        graphs, desc = make_workload(name, rank, backend)
        c = counts(graphs)
        return graphs, desc, {k: v * world for k, v in c.items()}
    allg: list = []
    for r in range(world):
        g, desc = make_workload(name, r, backend)
        allg += g
    parts = partition_graphs([graph_cost(g) for g in allg], world)
    return [allg[i] for i in parts[rank]], desc, counts(allg)


def train_labels(preds, seed: int):
    """labels = prediction + uniform noise (SURVEY.md §8d C5: +-0.1 eV/atom, +-0.01 eV/A, +-0.05 GPa, +-0.03 muB)"""
    gen = torch.Generator().manual_seed(seed)

    def noisy(v, amp):
        v = torch.as_tensor(np.asarray(v), dtype=torch.float32)
        return v + (torch.rand(v.shape, generator=gen) - 0.5) * 2 * amp

    return {"e": noisy([float(p["e"]) for p in preds], 0.1), "f": [noisy(p["f"], 0.01) for p in preds],
            "s": [noisy(p["s"], 0.05) for p in preds], "m": [noisy(p["m"], 0.03) for p in preds]}


def run_reference_train(args) -> None:
    """--impl reference --workload c5: one reference training step (trainer.py:398-411) on the host
    cores: oracle forward (train mode) -> CombinedLoss('em', MSE) -> backward -> torch Adam."""
    from oracle import chgnet_oracle as orc

    graphs, desc = make_workload("c5", 0, backend="numpy")  # numpy builder: the product .so is never mapped here
    sample = graphs[: max(1, min(len(graphs), args.cpu_sample if args.cpu_sample > 0 else 4))]
    w = orc.load_weights_npz(WEIGHTS)
    base = orc.predict_graph(w, sample, "efsm", batch_size=len(sample))
    lab = train_labels(base, 5)
    P = {k: torch.as_tensor(np.asarray(v)).float().requires_grad_(k != "composition_model.fc.weight") for k, v in w.items()}
    opt = torch.optim.Adam([v for v in P.values() if v.requires_grad], lr=1e-3)
    crit = torch.nn.MSELoss()

    def step():
        opt.zero_grad()
        out = orc.forward(P, sample, "efsm", train=True)
        loss = (crit(lab["e"], out["e"]) + crit(torch.cat(lab["f"]), torch.cat(out["f"]))
                + 0.1 * crit(torch.stack(lab["s"]), torch.stack(out["s"])) + 0.1 * crit(torch.cat(lab["m"]), torch.cat(out["m"])))
        loss.backward()
        opt.step()

    threads = pick_cpu_threads(step)
    for _ in range(max(1, args.warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = len(sample) / dt
    sdesc = f"first {len(sample)} graphs of the batch per step; {threads} of {os.cpu_count()} host threads (fastest of a 4..all sweep)"
    print(json.dumps({
        "impl": "reference", "metric": "train_structures_per_sec_EFSM", "value": value, "unit": "structures/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config("c5", desc, {k: v * int(os.environ.get("WORLD_SIZE", 1)) for k, v in counts(graphs).items()},
                               int(os.environ.get("WORLD_SIZE", 1)), task="train efsm"),
        "cpu_baseline": {"value": value, "unit": "structures/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sdesc},
        "e2e": {"value": value, "unit": "structures/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "product_so_mapped": product_so_mapped()}))


def run_train(args, rank: int, world: int, local_rank: int, light: bool = False):
    """--workload c5: one fine-tuning step per 'step' (forward, CombinedLoss, parameter gradients,
    one gradient all-reduce over NCCL, fused Adam, weight re-pack).

    ``light=True`` (the "collective" leg appended to a multi-GPU inference run): only the timed resident
    steps, with the all-reduce bracketed by its own CUDA events; returns a dict on every rank, prints nothing."""
    import contextlib
    import io

    import torch.distributed as dist

    from chgnet_b200.batch import build_batch
    from chgnet_b200.model import CHGNet
    from chgnet_b200.trainer import Trainer, loss_and_grads

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    with contextlib.redirect_stdout(io.StringIO()):
        model = CHGNet.from_file(WEIGHTS, version="0.3.0").to(dev)
    graphs, desc = make_workload("c5", rank)
    c = counts(graphs)
    base = model.predict_graph(graphs, task="efsm", batch_size=len(graphs))
    lab = train_labels(base, 5 + rank)
    trainer = Trainer(model, targets="efsm", criterion="MSE", learning_rate=1e-3)
    flush = L2Flush(dev)
    K = model._get_engine().K

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    batch = build_batch(graphs, dev, with_reverse=True)
    tg_dev = trainer._targets(lab, batch.atoms_per_graph, dev)

    ar_events: list = []

    def step_resident():
        engine = model._get_engine()  # re-packs the weights the previous Adam step changed
        report_, G = loss_and_grads(engine, batch, trainer.cfg, tg_dev, model.is_intensive, None)
        fg = trainer.flatten_packed_grads(G)
        if world > 1:
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            dist.all_reduce(fg)
            a1.record()
            ar_events.append((a0, a1, fg.numel() * fg.element_size()))
        trainer.step_count += 1
        K.adam_step(trainer.flat, fg, trainer.exp_avg, trainer.exp_avg_sq, trainer.lr, 0.9, 0.999, 1e-8, 0.0, trainer.step_count)
        trainer.refresh_packed_weights()
        return report_

    n_steps = min(args.steps, 5) if light else args.steps
    for _ in range(3 if light else max(args.warmup, 3)):
        flush()
        step_resident()
    barrier()
    ar_events.clear()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = K.launches
    elapsed_ms = 0.0
    for _ in range(n_steps):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rep_last = step_resident()
        e.record()
        e.synchronize()
        elapsed_ms += s.elapsed_time(e)
    barrier()
    launches = K.launches - launches0
    clocks = sampler.stop()
    ar_us = [a0.elapsed_time(a1) * 1e3 for a0, a1, _ in ar_events]
    t = torch.tensor([elapsed_ms, max(ar_us) if ar_us else 0.0, float(np.median(ar_us)) if ar_us else 0.0],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t[0].item()) / n_steps
    collective = None
    if world > 1:
        collective = {"op": "all_reduce(SUM) of the flat fp32 gradient buffer", "backend": "nccl", "bytes": int(ar_events[0][2]),
                      "us": round(float(t[2].item()), 1), "us_max": round(float(t[1].item()), 1),
                      "timing": "CUDA events around dist.all_reduce on the launching stream, median over steps, max over ranks "
                                "(includes waiting for the slowest rank's gradients)",
                      "train_ms_per_step": round(ms_per_step, 3), "train_structures_per_s": round(c["graphs"] * world / (ms_per_step * 1e-3), 1),
                      "steps": n_steps, "workload": f"c5: {desc}", "per_gpu": c}
    if light:
        return collective
    # host copy now: the end-to-end steps below train further.  The last timed step's loss report, its (all-reduced)
    # flat gradient and the parameters after its Adam update
    outputs = {"grad": trainer.flat_grad.cpu().numpy(), "params": trainer.flat.cpu().numpy(),
               **{k: np.float64(v) for k, v in rep_last.items() if not k.endswith("_size")}}

    # end to end: Trainer.train_step from host graphs + host labels, report read back every step
    targets = lab
    for _ in range(2):
        trainer.train_step(graphs, targets)
    h2d = int(build_batch(graphs, dev, with_reverse=True).h2d_bytes) + 4 * sum(int(v.numel()) for v in tg_dev.values())
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush()
        trainer.train_step(graphs, targets)
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item()) / args.steps
    if rank != 0:
        if world > 1:
            dist.barrier()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    # breakdown of one resident step (synchronised, outside the timed loops)
    from chgnet_b200.engine import EV_A3_TO_GPA
    from chgnet_b200.trainer import loss_and_seeds

    def tick():
        torch.cuda.synchronize()
        return time.perf_counter()

    t0 = tick()
    engine = model._get_engine()
    t1 = tick()
    o = engine.run(batch, need_grad=True, need_magmom=True, train=True)
    t2 = tick()
    engine.input_grads(o, record=True)
    t3 = tick()
    n_dev = torch.tensor(batch.atoms_per_graph, device=dev, dtype=torch.float64)
    preds = {"e": ((o.energy + o.e_ref) / n_dev).float(), "m": o.magmom, "f": o.force.float(),
             "s": (o.virial.view(-1, 3, 3) * (EV_A3_TO_GPA / batch.volume.double())[:, None, None]).float()}
    rep_, seeds = loss_and_seeds(K, trainer.cfg, preds, tg_dev, False)  # rank 0 only: no collective here
    t4 = tick()
    G = engine.param_grads(o, (seeds["e"] / n_dev.float()).contiguous(), seeds["m"], seeds["f"], seeds["s"])
    t5 = tick()
    fg = trainer.flatten_packed_grads(G)
    t6 = tick()
    breakdown = {"repack_weights_ms": (t1 - t0) * 1e3, "forward_ms": (t2 - t1) * 1e3, "force_pass_ms": (t3 - t2) * 1e3,
                 "loss_ms": (t4 - t3) * 1e3, "second_order_and_wgrads_ms": (t5 - t4) * 1e3,
                 "unpack_flatten_grads_ms": (t6 - t5) * 1e3}
    peaks, peak_kind = measured_peaks()
    sc_ms, sc_bytes = time_scatter_kernel(K, batch)
    achieved = sc_bytes / (sc_ms * 1e-3) / 1e9
    roofline = {"kernel": "segment_sum_kernel<128> (AtomConv scatter-reduce of the reverse pass)", "bound": "hbm", "achieved": round(achieved, 1),
                "peak": peaks["hbm_gbs"], "peak_kind": f"{peak_kind} copy bandwidth", "unit": "GB/s",
                "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": None, "us_per_launch": round(sc_ms * 1e3, 2),
                "algorithmic_bytes": sc_bytes, "bytes_formula": "512*E_d + 512*N + 4*(N+1)"}
    ek = EventKernels(K)
    from chgnet_b200.engine import Engine

    eng2 = Engine(model._get_engine().pw, ek)
    out2 = eng2.run(batch, need_grad=True, need_magmom=True, train=True)
    eng2.input_grads(out2, record=True)
    eng2.param_grads(out2, torch.ones(c["graphs"], device=dev), torch.ones(c["atoms"], device=dev),
                     torch.ones(c["atoms"], 3, device=dev), torch.ones(c["graphs"], 3, 3, device=dev))
    shares = ek.table()
    total = c["graphs"] * world
    print(json.dumps({
        "metric": "train_structures_per_sec_EFSM", "value": total / (ms_per_step * 1e-3), "unit": "structures/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config("c5", desc, {k: v * world for k, v in c.items()}, world, task="train efsm"),
        "train": {"collective": "one all-reduce of the flat gradient buffer per step",
                  "second_order": "tangent pass + reverse over (primal, tangent) for the force / stress loss terms"},
        "e2e": {"value": total / (e2e_ms * 1e-3), "unit": "structures/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 48, "api": "Trainer.train_step(list[CrystalGraph] on host, labels on host)"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": None, "collective": collective,
        "last_report": rep_last, "breakdown": breakdown, "kernel_shares": shares}), flush=True)
    if world > 1:
        dist.barrier()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: what the timed path returned in its last step, one `<name>.npy` per array (float64 stays float64,
    everything else is written as float32), so that two builds can be compared output for output on the same inputs."""
    out = {k: np.asarray(v, dtype=np.float64 if np.asarray(v).dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def counts(graphs):
    n = sum(int(g.atomic_number.shape[0]) for g in graphs)
    ed = sum(int(g.atom_graph.reshape(-1, 2).shape[0]) for g in graphs)
    a = sum(int(g.bond_graph.reshape(-1, 5).shape[0]) for g in graphs)
    return {"graphs": len(graphs), "atoms": n, "directed_edges": ed, "undirected_bonds": ed // 2, "angles": a}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int) -> None:
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.sm_max = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self) -> None:
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop_evt.wait(0.02)

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=1.0)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def pick_cpu_threads(fn, repeats: int = 3) -> int:
    """The torch CPU path does not scale to every core of a big host (tiny ops, OpenMP fork/join): time
    `fn` per candidate thread count (one warm call, then the best of `repeats` timed calls) and keep the
    fastest, so the CPU baseline is the reference at its best, not at `os.cpu_count()`."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        fn()  # warm
        dt = float("inf")
        for _ in range(max(1, repeats)):
            t0 = time.perf_counter()
            fn()
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# ------------------------------------------------------------------------------------------
def product_so_mapped() -> bool:
    """True if this process has the product's kernel library mapped (the reference arm must not)."""
    try:
        with open("/proc/self/maps") as f:
            return "libchgnet_b200" in f.read()
    except OSError:
        return False


REF_BUDGET_S = 900.0  # wall-clock the reference arm may spend on its warm-up + timed steps


def run_reference(args, rank: int, world: int) -> None:
    """--impl reference: the reference's CPU path (oracle port = the reference's torch ops) on the host
    cores.  Inputs are built with the numpy builder, so the product's .so is never mapped by this process.
    Each step is `predict_graph` over the FULL batch when warm-up + steps fit REF_BUDGET_S; otherwise over the
    largest leading power-of-two fraction that does (stated in `sample`)."""
    if rank != 0:
        return
    from oracle import chgnet_oracle as orc

    graphs, desc = make_workload(args.workload, 0, backend="numpy")
    whole = {k: v * world for k, v in counts(graphs).items()} if (world == 1 or args.workload in ("c1", "c4")) else None
    if whole is None:
        allg = list(graphs)
        for r in range(1, world):
            allg += make_workload(args.workload, r, backend="numpy")[0]
        whole = counts(allg)
    w = orc.load_weights_npz(WEIGHTS)
    if args.workload == "c4":
        from chgnet_b200 import graphgen

        z, frac, lat = graphgen.limno2_structure((5, 4, 3), 0.02, 4000)
        sample = [graphgen.make_crystal_graph(z, frac, lat, backend="numpy")]
        probe = sample
        desc_s = "LiMnO2 5x4x3 supercell (480 atoms) - largest cell timed on the CPU; value scaled by atoms"
    else:
        probe = graphs[:2]
    threads = pick_cpu_threads(lambda: orc.predict_graph(w, probe, "efs", batch_size=len(probe)))
    if args.workload != "c4":
        # size the per-step sample from a measured rate: full batch if (warmup + steps) of it fit the budget
        n_probe = min(len(graphs), 8)
        orc.predict_graph(w, graphs[:n_probe], "efs", batch_size=n_probe)
        t0 = time.perf_counter()
        orc.predict_graph(w, graphs[:n_probe], "efs", batch_size=n_probe)
        per_graph = (time.perf_counter() - t0) / n_probe
        n = len(graphs) if args.cpu_sample <= 0 else min(len(graphs), args.cpu_sample)
        while n > 8 and per_graph * n * (args.steps + args.warmup) > REF_BUDGET_S:
            n = max(8, n // 2)
        sample = graphs[:n]
        why = ("--cpu-sample" if args.cpu_sample > 0 and n == args.cpu_sample else
               f"the full batch would exceed {REF_BUDGET_S:.0f} s for {args.steps}+{args.warmup} steps at {1.0 / per_graph:.1f} structures/s")
        desc_s = ("the full batch per step" if n == len(graphs) else
                  f"first {n} of {len(graphs)} graphs per step ({n / len(graphs):.3f} of the batch: {why})")
    desc_s += (f"; {threads} of {os.cpu_count()} host threads (fastest of a 4..all sweep, best of 3 per candidate); "
               "16 graphs per forward (the reference's default batch_size)")
    # predict_graph's batching loop (model.py:634-645) at the reference's own default batch_size = 16 (model.py:601): the CPU
    # path is FASTEST there (measured on the pool's hosts: 17 structures/s at 8-16 graphs per forward, 5 at 64)
    bs = min(len(sample), 16)
    for _ in range(args.warmup):
        orc.predict_graph(w, sample, "efs", batch_size=bs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.predict_graph(w, sample, "efs", batch_size=bs)
    dt = (time.perf_counter() - t0) / args.steps
    c = counts(sample)
    value = c["graphs"] / dt
    if args.workload == "c4":
        value = (c["atoms"] / dt) / counts(graphs)["atoms"]  # 10k-atom structures/s at the same atoms/s
    line = {
        "impl": "reference", "metric": "structures_per_sec_EFS", "value": value, "unit": "structures/s",
        "atoms_per_s": c["atoms"] / dt, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": bench_config(args.workload, desc, whole, world),
        "cpu_baseline": {"value": value, "unit": "structures/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": desc_s, "sample_counts": c},
        "e2e": {"value": value, "unit": "structures/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "product_so_mapped": product_so_mapped(),
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
class L2Flush:
    """Evicts everything of ours from the 126 MB L2 between timed iterations: writes a 256 MiB
    buffer (the rule of the task statement), then streams a second 256 MiB buffer through with a
    read so that the cache is left holding CLEAN lines — otherwise the timed kernel also pays
    for the write-back of the flush buffer's dirty lines."""

    def __init__(self, dev) -> None:
        self.w = torch.empty(L2_FLUSH_BYTES // 4, device=dev)
        self.r = torch.zeros(L2_FLUSH_BYTES // 4, device=dev)
        self.sink = torch.zeros((), device=dev)

    def __call__(self) -> None:
        self.w.zero_()
        self.sink.copy_(self.r.sum())


def time_scatter_kernel(K, batch, n_iter: int = 20, width: int = 128):
    """The AtomConv scatter-reduce alone: chg_segment_sum over centre-sorted rows, CUDA events on the launching stream, L2
    flushed.  width = 128: the reverse-pass call (dE/dpre rows -> per-atom sums, the scatter that still runs as its own
    kernel); width = 64: the forward message sum (now fused into gated_ws_fwd_kernel, kept for continuity with round 1)."""
    dev = batch.z.device
    msg = torch.randn(batch.n_edges, width, device=dev)
    out = torch.empty(batch.n_atoms, width, device=dev)
    flush = L2Flush(dev)
    for _ in range(3):
        K.segment_sum(msg, None, batch.ptr_c, 0, out)
    total = 0.0
    for _ in range(n_iter):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        K.segment_sum(msg, None, batch.ptr_c, 0, out)
        e.record()
        e.synchronize()
        total += s.elapsed_time(e)
    ms = total / n_iter
    alg_bytes = 4 * width * batch.n_edges + 4 * width * batch.n_atoms + 4 * (batch.n_atoms + 1)
    return ms, alg_bytes


class EventKernels:
    """Wraps the kernel binding with per-call CUDA events (used OUTSIDE the timed region)."""

    def __init__(self, inner) -> None:
        self._inner, self.records = inner, []

    def __getattr__(self, name):
        attr = getattr(self._inner, name)
        if not callable(attr) or name.startswith("_"):
            return attr

        def timed(*a):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            attr(*a)
            e.record()
            self.records.append((name, s, e))

        return timed

    def table(self):
        torch.cuda.synchronize()
        agg: dict[str, list] = {}
        for name, s, e in self.records:
            agg.setdefault(name, [0.0, 0])
            agg[name][0] += s.elapsed_time(e)
            agg[name][1] += 1
        tot = sum(v[0] for v in agg.values()) or 1.0
        return {k: {"ms": round(v[0], 4), "calls": v[1], "share": round(v[0] / tot, 4)}
                for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}


def infer_leg(model, graphs, dev, local_rank: int, world: int, steps: int, warmup: int, replay: bool = False) -> dict:
    """Times one workload two ways: the kernel path on a resident batch descriptor (CUDA events per step, L2
    flushed between steps) and `CHGNet.predict_graph` from host CrystalGraphs (wall clock per step, device
    synchronised on both sides; host packing, H2D, CSR build, kernels, D2H inside).  Max over ranks."""
    import torch.distributed as dist

    from chgnet_b200.batch import build_batch
    from chgnet_b200.engine import EV_A3_TO_GPA

    K = model._get_engine().K
    flush = L2Flush(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    batch = build_batch(graphs, dev, with_reverse=True)
    native = model._get_native()  # the product's inference path: ONE chg_forward call per step

    def step_resident():
        # replay: the resident descriptor is evaluated through NativeForward.replay (one captured CUDA graph of chg_forward)
        out = native.replay(batch, need_grad=True) if replay else native(batch, need_grad=True)
        scale = EV_A3_TO_GPA / batch.volume.to(torch.float64)
        stress = (out["virial"].view(-1, 3, 3) * scale[:, None, None]).to(torch.float32)
        return out["energy"], out["force"].to(torch.float32), stress

    for _ in range(max(warmup, 3)):
        flush()
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = K.launches
    elapsed_ms = 0.0
    t_wall0 = time.perf_counter()
    for _ in range(steps):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        last = step_resident()
        e.record()
        e.synchronize()
        elapsed_ms += s.elapsed_time(e)
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    launches = K.launches - launches0
    clocks = sampler.stop()
    # host copy now: a replayed CUDA graph reuses its output tensors, and later legs replay it
    outputs = {name: t.cpu().numpy() for name, t in zip(("energy", "force", "stress"), last)}

    # ---------------- end to end through the public API ----------------
    def step_e2e():
        return model.predict_graph(graphs, task="efs", batch_size=len(graphs))

    for _ in range(2):
        preds = step_e2e()
    d2h = sum(int(v.nbytes) for p in preds for v in p.values())
    h2d = int(model.last_batch.h2d_bytes)
    barrier()
    e2e_ms = 0.0
    for _ in range(steps):
        flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        preds = step_e2e()
        torch.cuda.synchronize()
        e2e_ms += (time.perf_counter() - t0) * 1e3
    t = torch.tensor([elapsed_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"ms_per_step": float(t[0].item()) / steps, "e2e_ms_per_step": float(t[1].item()) / steps, "launches": int(launches),
            "clocks": clocks, "wall_ms": wall_ms, "h2d": h2d, "d2h": d2h, "preds": preds, "batch": batch, "outputs": outputs}


def md_leg(model, dev, steps: int = 20) -> dict:
    """NVE molecular dynamics of the 10,000-atom cell (BASELINE configs[3] is "one MD step"): device-resident driver
    (positions / velocities / forces on the GPU, device graph builder with a Verlet skin, one CUDA graph per step) next to
    the host-driven loop the reference's CHGNetCalculator implies (host graph build -> H2D -> model -> D2H every step)."""
    from chgnet_b200 import graphgen
    from chgnet_b200.dynamics import Atoms, CHGNetCalculator, VelocityVerlet
    from chgnet_b200.dynamics_device import DeviceMD

    z, frac, lat = graphgen.limno2_structure((10, 5, 25), 0.02, 4000)
    pos = frac @ lat
    def run_device(skin):
        md = DeviceMD(model, z, pos, lat, timestep=2.0, skin=skin)
        md.set_temperature(300.0, seed=1)
        md.run(5, log_every=0)
        torch.cuda.synchronize()
        md.t_rebuild = md.t_capture = 0.0
        b0 = md.n_builds
        t0 = time.perf_counter()
        md.run(steps, log_every=0)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        return {"ms_per_step": round(dt * 1e3, 3), "steps_per_s": round(1.0 / dt, 2), "steps": steps, "skin_A": md.skin,
                "graph_rebuilds": md.n_builds - b0, "model_edges": int(md.batch.n_edges), "model_angles": int(md.batch.n_angles),
                "host_s_in_rebuilds": round(md.t_rebuild, 4), "host_s_in_captures": round(md.t_capture, 4),
                "e_total_eV": md.potential_energy + md.kinetic_energy}

    dev_exact = run_device(0.0)
    dev_exact["what"] = ("DeviceMD(skin=0): kick+drift -> chg_graph_build_device + chg_build_csr (exact lists, every step) -> "
                         "chg_forward -> kick; positions / velocities / forces never leave the device")
    dev_skin = run_device(0.5)
    dev_skin["what"] = "DeviceMD(skin=0.5): lists with cutoffs + 0.5 A reused until an atom moved 0.25 A; the step is one CUDA graph replay"
    host = VelocityVerlet(Atoms(z, pos, lat), CHGNetCalculator(model=model, on_isolated_atoms="ignore"), timestep=2.0)
    host.set_temperature(300.0, seed=1)
    host.run(2)
    t0 = time.perf_counter()
    host.run(5)
    dt_host = (time.perf_counter() - t0) / 5
    return {"atoms": int(len(z)), "timestep_fs": 2.0, "temperature_K": 300.0, "device_driver": dev_exact, "device_driver_skin": dev_skin,
            "host_driver": {"ms_per_step": round(dt_host * 1e3, 3), "steps_per_s": round(1.0 / dt_host, 2), "steps": 5,
                            "what": "CHGNetCalculator loop (the reference's structure, dynamics.py:129-181): host graph build "
                                    "(native C++), H2D, chg_forward, D2H, numpy integrator"}}


def scatter_roofline(K, batch, workload: str, dev) -> dict:
    """Roofline record of the AtomConv scatter-reduce kernel at this batch's size (DESIGN.md §4)."""
    peaks, peak_kind = measured_peaks()
    sc_ms, sc_bytes = time_scatter_kernel(K, batch, width=128)
    achieved = sc_bytes / (sc_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "scatter_traffic.json")
    if os.path.exists(tpath):  # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu capture
        with open(tpath) as f:
            traffic = json.load(f).get(workload + "_w128", {}).get("dram_bytes_per_launch")
    ms64, b64 = time_scatter_kernel(K, batch, width=64)
    return {"kernel": "segment_sum_kernel<128> (AtomConv scatter-reduce of the reverse pass: dE/dpre rows -> atoms)", "bound": "hbm",
            "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"], "peak_kind": f"{peak_kind} copy bandwidth",
            "unit": "GB/s", "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": traffic,
            "us_per_launch": round(sc_ms * 1e3, 2), "algorithmic_bytes": sc_bytes,
            "bytes_formula": "512*E_d + 512*N + 4*(N+1)",
            "forward_message_sum_w64": {"us_per_launch": round(ms64 * 1e3, 2), "algorithmic_bytes": b64,
                                        "frac": round(b64 / (ms64 * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                                        "note": "round-1 roofline kernel; in the default forward this sum is now fused into "
                                                "gated_ws_fwd_kernel (the message never reaches HBM)"}}


def bind_to_gpu_numa_node(local_rank: int):
    """One process per GPU: keep this process (and the packer's worker threads it creates later) on the CPUs NVML reports as
    local to its GPU, so that the pinned staging buffers and the threads that fill them sit on the GPU's NUMA node (what
    `numactl --cpunodebind` does in a deployment).  Returns (previous mask, description) or (None, why not); the CPU-baseline
    leg restores the previous mask.  CHGNET_BENCH_BIND=0 disables it."""
    if os.environ.get("CHGNET_BENCH_BIND", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return None, "disabled"
    try:
        import pynvml

        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        index = int(visible.split(",")[local_rank]) if visible and visible.split(",")[local_rank].isdigit() else local_rank
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        prev = os.sched_getaffinity(0)
        cpus &= prev
        if not cpus or cpus == prev:
            return None, f"NVML reports no narrower CPU set for GPU {index} ({len(prev)} CPUs allowed)"
        os.sched_setaffinity(0, cpus)
        return prev, f"{len(cpus)} of {len(prev)} CPUs (local to GPU {index}: {min(cpus)}..{max(cpus)})"
    except Exception as exc:  # noqa: BLE001  (no NVML / no permission: run unbound)
        return None, f"unavailable: {exc!r}"[:160]


def run_ours(args, rank: int, world: int, local_rank: int) -> None:
    import contextlib
    import io

    import torch.distributed as dist

    from chgnet_b200.batch import build_batch
    from chgnet_b200.engine import Engine
    from chgnet_b200.model import CHGNet

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    prev_affinity, binding = bind_to_gpu_numa_node(local_rank)
    with contextlib.redirect_stdout(io.StringIO()):
        model = CHGNet.from_file(WEIGHTS, version="0.3.0").to(dev).eval()
    graphs, desc, whole = sharded_workload(args.workload, rank, world)
    c = counts(graphs)
    engine = model._get_engine()
    K = engine.K

    if args.scatter_only:  # ncu capture target: only the AtomConv scatter-reduce launches
        batch = build_batch(graphs, dev, with_reverse=True)
        ms, nbytes = time_scatter_kernel(K, batch, n_iter=5)
        print(json.dumps({"scatter_only": True, "us_per_launch": ms * 1e3, "algorithmic_bytes": nbytes}))
        return

    leg = infer_leg(model, graphs, dev, local_rank, world, args.steps, args.warmup, replay=args.graph_replay)
    batch = leg["batch"]
    ms_per_step, e2e_ms_per_step = leg["ms_per_step"], leg["e2e_ms_per_step"]

    # ---------------- the same resident step replayed as ONE CUDA graph (NativeForward.replay) ----------------
    graph_replay = None
    if not args.graph_replay and world == 1:  # single-GPU records only
        try:
            nat, flush_r = model._get_native(), L2Flush(dev)
            for _ in range(3):  # eager, capture, first replay
                nat.replay(batch, need_grad=True)
            torch.cuda.synchronize()
            tot = 0.0
            for _ in range(args.steps):
                flush_r()
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record()
                nat.replay(batch, need_grad=True)
                e_.record()
                e_.synchronize()
                tot += s_.elapsed_time(e_)
            graph_replay = {"ms_per_step": round(tot / args.steps, 4), "structures_per_s": round(len(graphs) / (tot / args.steps * 1e-3), 1),
                            "what": "this rank's resident batch, chg_forward captured once and replayed (one graph launch per step); "
                                    "what CHGNet.static_evaluator and DeviceMD use; NOT the headline value"}
        except Exception as exc:  # reported, never fatal for the bench line
            graph_replay = {"unavailable": repr(exc)[:200]}

    # ---------------- N > 1: the path's one collective (c5 fine-tuning step), every rank ----------------
    collective = None
    if world > 1 and not args.no_collective:
        collective = run_train(args, rank, world, local_rank, light=True)

    if rank != 0:
        if world > 1:
            dist.barrier()  # wait for rank 0's extra legs (roofline, shares, c4, CPU baseline)
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, leg["outputs"])
    # e2e breakdown (one synchronised pass, outside the timed loops)
    native = model._get_native()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bb = build_batch(graphs, dev, with_reverse=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    oo = native(bb, need_grad=True)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    _ = (oo["energy"].cpu(), oo["force"].to(torch.float32).cpu(), oo["virial"].cpu())
    t3 = time.perf_counter()
    breakdown = {"pack_h2d_csr_ms": (t1 - t0) * 1e3, "kernels_ms": (t2 - t1) * 1e3, "d2h_ms": (t3 - t2) * 1e3}
    # ---------------- roofline of the AtomConv scatter kernel ----------------
    roofline = scatter_roofline(K, batch, args.workload, dev)
    peaks, _ = measured_peaks()
    # the same kernel at the AtomConv size of the 10,000-atom cell (84 edges per atom), on
    # synthetic uniform segments - the size the north-star's >= 50 % target is quoted for
    if args.workload != "c4":
        class _B:  # minimal stand-in carrying the three fields time_scatter_kernel reads
            z = batch.z
            n_atoms, n_edges = 10000, 840000
            ptr_c = (torch.arange(10001, device=dev, dtype=torch.int32) * 84).contiguous()
        ms10, b10 = time_scatter_kernel(K, _B, width=128)
        roofline["at_10k_atoms"] = {"us_per_launch": round(ms10 * 1e3, 2), "algorithmic_bytes": b10,
                                    "achieved": round(b10 / (ms10 * 1e-3) / 1e9, 1),
                                    "frac": round(b10 / (ms10 * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                                    "input": "synthetic: 10,000 segments x 84 rows x 512 B"}
    # per-kernel shares (own events, outside the timed region)
    ek = EventKernels(K)
    Engine(engine.pw, ek).run(batch, need_grad=True)
    shares = ek.table()
    fa = shares.get("atom_conv_fused")
    if fa:
        # the forward AtomConv scatter now lives inside the fused tile kernel: its compulsory traffic (SURVEY.md §8d "fully fused
        # AtomConv": 268 E_d + 512 N) plus the 512 B / edge of p kept for the reverse pass, against the same HBM peak
        us = fa["ms"] / fa["calls"] * 1e3
        nb = (268 + 512) * c["directed_edges"] + 512 * c["atoms"]
        roofline["fused_forward_atom_conv"] = {
            "kernel": "gated_ws_fwd_kernel<ATOM> + seg_stitch_kernel (message + aggregation, tcgen05)", "us_per_launch": round(us, 2),
            "compulsory_bytes": nb, "bytes_formula": "(268 + 512 saved p) * E_d + 512 * N",
            "achieved": round(nb / (us * 1e-6) / 1e9, 1), "frac": round(nb / (us * 1e-6) / 1e9 / peaks["hbm_gbs"], 4),
            "note": "latency-bound (gathers + MUFU), not bandwidth-bound: see profiles/ for tensor-pipe % and DRAM bytes"}

    # ---------------- the 10,000-atom cell (BASELINE configs[3]) as an extra key ----------------
    c4 = None
    if args.workload in ("c2", "c3") and not args.no_c4:
        g4, d4 = make_workload("c4", 0)
        c4c = counts(g4)
        l4 = infer_leg(model, g4, dev, local_rank, 1, min(args.steps, 10), 3)
        c4 = {"workload": f"c4: {d4}", "counts": c4c, "ms_per_step": round(l4["ms_per_step"], 4),
              "atoms_per_s": round(c4c["atoms"] / (l4["ms_per_step"] * 1e-3), 1),
              "structures_per_s": round(1e3 / l4["ms_per_step"], 2), "gpu_launches_per_step": l4["launches"] // min(args.steps, 10),
              "e2e": {"ms_per_step": round(l4["e2e_ms_per_step"], 4), "atoms_per_s": round(c4c["atoms"] / (l4["e2e_ms_per_step"] * 1e-3), 1),
                      "h2d_bytes_per_step": l4["h2d"], "d2h_bytes_per_step": l4["d2h"],
                      "api": "CHGNet.predict_graph(CrystalGraph on host, task='efs')"},
              "roofline": scatter_roofline(K, l4["batch"], "c4", dev), "clocks": l4["clocks"], "n_gpus": 1,
              "note": "one structure does not shard: rank 0 alone (replicas only, DESIGN.md §7)"}
        try:  # the same structure through predict_structure: graph built ON THE DEVICE, only z / frac / lattice cross PCIe
            from chgnet_b200 import graphgen as _gg

            z4, f4, l4m = _gg.limno2_structure((10, 5, 25), 0.02, 4000)
            for _ in range(2):
                model.predict_structure((z4, f4, l4m), task="efs")
            tt = 0.0
            flush4 = L2Flush(dev)
            for _ in range(5):
                flush4()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                model.predict_structure((z4, f4, l4m), task="efs")
                torch.cuda.synchronize()
                tt += time.perf_counter() - t0
            c4["e2e_from_structure"] = {"ms_per_step": round(tt / 5 * 1e3, 4), "atoms_per_s": round(c4c["atoms"] / (tt / 5), 1),
                                        "over_kernel_path": round(tt / 5 * 1e3 / l4["ms_per_step"], 3),
                                        "h2d_bytes_per_step": int(c4c["atoms"] * (4 + 24) + 72), "d2h_bytes_per_step": l4["d2h"],
                                        "api": "CHGNet.predict_structure((Z, frac, lattice), task='efs'): chg_graph_build_device + "
                                               "chg_build_csr + chg_forward"}
        except Exception as exc:
            c4["e2e_from_structure"] = {"unavailable": repr(exc)[:300]}
        if not args.no_md:
            try:
                c4["md"] = md_leg(model, dev)
            except Exception as exc:  # reported, never fatal for the bench line
                c4["md"] = {"unavailable": repr(exc)[:300]}

    # ---------------- CPU baseline + parity: oracle port on the host cores ----------------
    cpu = None
    torch_cuda = None
    parity = None
    if not args.no_cpu_baseline:
        from oracle import chgnet_oracle as orc

        if prev_affinity is not None:  # the CPU baseline may use every core of the host
            os.sched_setaffinity(0, prev_affinity)
        w = orc.load_weights_npz(WEIGHTS)
        n_s = min(len(graphs), args.cpu_sample if args.cpu_sample > 0 else 8)
        if args.workload == "c4":
            from chgnet_b200 import graphgen

            z, frac, lat = graphgen.limno2_structure((5, 4, 3), 0.02, 4000)
            sample = [graphgen.make_crystal_graph(z, frac, lat)]
            sdesc = "LiMnO2 5x4x3 (480 atoms), 1 warm-up + 2 timed; structures/s scaled by atoms to the 10,000-atom cell"
            gpu_sample = model.predict_graph(sample, task="efs", batch_size=1)
        else:
            sample = graphs[:n_s]
            sdesc = f"first {len(sample)} graphs of the batch, 1 warm-up + 2 timed predict_graph(task='efs') calls"
            gpu_sample = leg["preds"][:n_s]  # what the timed e2e call returned for the same graphs
        probe = sample[:2]
        threads = pick_cpu_threads(lambda: orc.predict_graph(w, probe, "efs", batch_size=len(probe)))
        sdesc += f"; {threads} of {os.cpu_count()} host threads (fastest of a 4..all sweep, best of 3 per candidate)"
        orc.predict_graph(w, sample, "efs", batch_size=len(sample))
        t0 = time.perf_counter()
        for _ in range(2):
            ref_sample = orc.predict_graph(w, sample, "efs", batch_size=len(sample))
        dt = (time.perf_counter() - t0) / 2
        cs = counts(sample)
        v = cs["graphs"] / dt if args.workload != "c4" else (cs["atoms"] / dt) / c["atoms"]
        cpu = {"value": v, "unit": "structures/s", "atoms_per_s": cs["atoms"] / dt, "cores": torch.get_num_threads(),
               "kind": "port", "sample": sdesc}
        # parity of the timed GPU outputs against the CPU baseline's outputs on the same graphs
        def worst(k):
            return max(float(np.max(np.abs(np.asarray(a[k], np.float64) - np.asarray(b[k], np.float64)))) for a, b in zip(gpu_sample, ref_sample))
        parity = {"e": worst("e"), "f": worst("f"), "s": worst("s"), "unit": "eV/atom, eV/A, GPa (max abs)",
                  "vs": f"oracle port (fp32 torch CPU = the reference's arithmetic) on {len(sample)} graph(s) of this run",
                  "tolerance": {"e": 1e-4, "f": 1e-3, "s": 1e-3},
                  "ok": bool(worst("e") < 1e-4 and worst("f") < 1e-3 and worst("s") < 1e-3)}
        # the realistic incumbent (SURVEY.md §8d): the reference's torch ops on the SAME B200 (stock PyTorch CUDA)
        if args.workload != "c4":
            try:
                for _ in range(2):
                    orc.predict_graph(w, graphs, "efs", batch_size=len(graphs), device=dev)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    orc.predict_graph(w, graphs, "efs", batch_size=len(graphs), device=dev)
                torch.cuda.synchronize()
                dtc = (time.perf_counter() - t0) / 3
                torch_cuda = {"value": c["graphs"] / dtc, "unit": "structures/s", "ms_per_step": dtc * 1e3,
                              "what": "oracle port = the reference's torch ops and per-graph batching loop, stock PyTorch "
                                      "CUDA on the same B200, fp32, host graphs in / numpy out, this rank's share (compare with e2e / n_gpus)"}
            except Exception as exc:  # reported, never fatal for the bench line
                torch_cuda = {"unavailable": repr(exc)[:200]}

    total_graphs = whole["graphs"]
    value = total_graphs / (ms_per_step * 1e-3)
    cfg = bench_config(args.workload, desc, whole, world)
    line = {
        "metric": "structures_per_sec_EFS", "value": value, "unit": "structures/s",
        "atoms_per_s": whole["atoms"] / (ms_per_step * 1e-3),
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg, "rank0_share": c, "cpu_binding": binding,
        "engine": "native chg_forward (one C call per step); kernel_shares via the Python schedule of the same kernels",
        "e2e": {"value": total_graphs / (e2e_ms_per_step * 1e-3), "unit": "structures/s",
                "ms_per_step": e2e_ms_per_step, "h2d_bytes_per_step": leg["h2d"], "d2h_bytes_per_step": leg["d2h"],
                "api": "CHGNet.predict_graph(list[CrystalGraph] on host, task='efs')", "breakdown": breakdown,
                "over_kernel_path": round(e2e_ms_per_step / ms_per_step, 3)},
        "gpu_launches": leg["launches"], "wall_ms_timed_region": leg["wall_ms"],
        "clocks": leg["clocks"], "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "c4": c4, "collective": collective, "graph_replay": graph_replay,
        "torch_cuda_baseline": torch_cuda, "kernel_shares": shares,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("CHGNET_BENCH_WORKLOAD", "c3"), choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="reference arm: graphs per step (0 = as many as fit the time budget); cpu_baseline leg of the product arm: 8 when 0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the 10,000-atom extra leg of a c2 / c3 run")
    ap.add_argument("--no-collective", action="store_true", help="N > 1: skip the c5 all-reduce leg")
    ap.add_argument("--no-md", action="store_true", help="skip the MD sub-leg of the c4 extra leg")
    ap.add_argument("--graph-replay", action="store_true", help="kernel-path leg: replay one captured CUDA graph of chg_forward per step")
    ap.add_argument("--scatter-only", action="store_true", help="run only the AtomConv scatter kernel timing (ncu target)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                    "(inference: energy, force, stress; c5: loss terms, grad, params); at N > 1, rank 0's share")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.scatter_only):
        ap.error("--dump-outputs applies to the product arm's timed path (--impl ours, without --scatter-only)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if args.workload == "c5":
            if rank == 0:
                run_reference_train(args)
            return
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; the hot path has no CPU implementation")
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        (run_train if args.workload == "c5" else run_ours)(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
