"""``CHGNet`` — drop-in model API over the B200 kernel engine.

Mirrors the public surface of the reference class (reference
chgnet/model/model.py:35-745): constructor keywords, ``forward`` (330-387),
``predict_graph`` (593-665), ``predict_structure`` (544-591), ``as_dict / todict /
from_dict / from_file / load`` (667-745), the returned dict layout, exception types
and messages.  Parameters are registered under the reference's ``state_dict`` names
(SURVEY.md §8 a-0), so reference checkpoints load unchanged and ``state_dict()`` can
be handed back to the reference.

The arithmetic is NOT torch: ``forward`` builds one :class:`DeviceBatch` and runs the
kernels through the C ABI — inference as ONE native call (``chg_forward``,
:mod:`chgnet_b200.native`), training through the schedule of :mod:`chgnet_b200.engine`
(``e / f / s / m`` then carry autograd history to the parameters).  No CPU path.

Limits (raise, never fall back): feature dims must be 64, GatedMLP hidden dims 64 (conv) /
0 (angle), layer- or no normalisation, ``mlp_first=True``.
"""
from __future__ import annotations

import math
import os
import warnings
from collections.abc import Sequence
from typing import Any, get_args

import numpy as np
import torch
from torch import Tensor, nn

from chgnet_b200 import PredTask
from chgnet_b200.batch import DeviceBatch, build_batch
from chgnet_b200.engine import EV_A3_TO_GPA, Engine
from chgnet_b200.graph import CrystalGraph, is_graph_like
from chgnet_b200.weights import pack_weights, unpack_grads

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)

_CHECKPOINTS = {
    "0.3.0": "0.3.0/chgnet_0.3.0_e29f68s314m37.pth.tar",
    "0.2.0": "0.2.0/chgnet_0.2.0_e30f77s348m32.pth.tar",
    "r2scan": "r2scan/chgnet_r2scan_transfer_learning_e15f36s161m23.pth.tar",
}


# --------------------------------------------------------------------------
# parameter tree with the reference's names
# --------------------------------------------------------------------------
def _mlp_linear_indices(hidden: Sequence[int] | int | None) -> tuple[list[int], int]:
    """Indices of the Linear layers inside the reference ``MLP.layers`` Sequential
    (reference chgnet/model/functions.py:71-92): hidden Linear positions, last Linear."""
    if hidden is None or hidden == 0:
        return [], 1
    if isinstance(hidden, int):
        return [0], 3
    n = len(hidden)
    return [2 * i for i in range(n)], 2 * n + 1


def _param_specs(a: dict) -> dict[str, tuple[tuple[int, ...], str]]:
    """name -> (shape, init kind) for every parameter of the architecture."""
    A, Bd, An = a["atom_fea_dim"], a["bond_fea_dim"], a["angle_fea_dim"]
    R, NA, n_conv = a["num_radial"], a["num_angular"], a["n_conv"]
    if NA % 2 != 1:
        raise ValueError(f"num_angular={NA} must be an odd integer")  # encoders.py:127-128
    specs: dict[str, tuple[tuple[int, ...], str]] = {}

    def lin(name, out_d, in_d, bias=True):
        specs[f"{name}.weight"] = ((out_d, in_d), "linear")
        if bias:
            specs[f"{name}.bias"] = ((out_d,), f"bias:{in_d}")

    def norm(name, dim, kind):
        if kind == "layer":
            specs[f"{name}.weight"] = ((dim,), "ones")
            specs[f"{name}.bias"] = ((dim,), "zeros")
        elif kind is not None:
            raise NotImplementedError(f"normalisation {kind!r} is not supported by chgnet_b200 (use 'layer' or None)")

    def gated(prefix, in_d, out_d, hidden):
        hid_idx, last = _mlp_linear_indices(hidden)
        hl = [hidden] if isinstance(hidden, int) and hidden else (list(hidden) if hidden else [])
        for br in ("mlp_core", "mlp_gate"):
            d = in_d
            for i, h in zip(hid_idx, hl):
                lin(f"{prefix}.{br}.layers.{i}", h, d)
                d = h
            lin(f"{prefix}.{br}.layers.{last}", out_d, d)
        norm(f"{prefix}.bn1", out_d, a["gMLP_norm"])
        norm(f"{prefix}.bn2", out_d, a["gMLP_norm"])

    if a.get("composition_model") is not None:
        specs["composition_model.fc.weight"] = ((1, 94), "atomref")
    specs["atom_embedding.embedding.weight"] = ((94, A), "normal")
    specs["bond_basis_expansion.rbf_expansion_ag.frequencies"] = ((R,), "rbf")
    specs["bond_basis_expansion.rbf_expansion_bg.frequencies"] = ((R,), "rbf")
    lin("bond_embedding", Bd, R, bias=False)
    lin("bond_weights_ag", A, R, bias=False)
    lin("bond_weights_bg", Bd, R, bias=False)
    specs["angle_basis_expansion.fourier_expansion.frequencies"] = (((NA - 1) // 2,), "fourier")
    lin("angle_embedding", An, NA, bias=False)
    for t in range(n_conv):
        gated(f"atom_conv_layers.{t}.twoBody_atom", 2 * A + Bd, A, a["atom_conv_hidden_dim"])
        lin(f"atom_conv_layers.{t}.mlp_out.layers.1", A, A, bias=a["mlp_out_bias"])
        norm(f"atom_conv_layers.{t}.atom_norm", A, a["conv_norm"])
    for t in range(n_conv - 1):
        if a["update_bond"]:
            gated(f"bond_conv_layers.{t}.twoBody_bond", A + 2 * Bd + An, Bd, a["bond_conv_hidden_dim"])
            lin(f"bond_conv_layers.{t}.mlp_out.layers.1", Bd, Bd, bias=a["mlp_out_bias"])
            norm(f"bond_conv_layers.{t}.bond_norm", Bd, a["conv_norm"])
        if a["update_angle"]:
            gated(f"angle_layers.{t}.twoBody_bond", A + 2 * Bd + An, An, a["angle_layer_hidden_dim"])
            norm(f"angle_layers.{t}.angle_norm", An, a["conv_norm"])
    lin("site_wise", 1, A)
    norm("readout_norm", A, a["readout_norm"])
    hid_idx, last = _mlp_linear_indices(a["mlp_hidden_dims"])
    hl = a["mlp_hidden_dims"]
    hl = [hl] if isinstance(hl, int) else list(hl)
    d = A
    for i, h in zip(hid_idx, hl):
        lin(f"mlp.layers.{i}", h, d)
        d = h
    lin(f"mlp.layers.{last}", 1, d)
    return specs


def _atomref_table(name: str) -> Tensor:
    path = os.path.join(_HERE, "atomref.npz")
    key = name
    if os.path.exists(path):
        with np.load(path) as f:
            if key in f.files:
                return torch.from_numpy(f[key].astype(np.float32)).reshape(1, 94)
    warnings.warn(f"AtomRef table {name!r} is not bundled; composition energies start at zero", stacklevel=3)
    return torch.zeros(1, 94)


def _init_param(shape, kind: str, a: dict) -> Tensor:
    if kind == "linear":
        bound = 1.0 / math.sqrt(shape[1])
        return torch.empty(shape).uniform_(-bound, bound)
    if kind.startswith("bias:"):
        bound = 1.0 / math.sqrt(int(kind.split(":")[1]))
        return torch.empty(shape).uniform_(-bound, bound)
    if kind == "ones":
        return torch.ones(shape)
    if kind == "zeros":
        return torch.zeros(shape)
    if kind == "normal":
        return torch.randn(shape)
    if kind == "rbf":  # basis.py:74-80
        return math.pi * torch.arange(1, shape[0] + 1, dtype=torch.float32)
    if kind == "fourier":  # basis.py:23-27
        return torch.arange(1, shape[0] + 1, dtype=torch.float32)
    if kind == "atomref":
        cm = a.get("composition_model")
        return _atomref_table(cm if isinstance(cm, str) else "MPtrj")
    raise AssertionError(kind)


class _ParamGradBridge(torch.autograd.Function):
    """Joins the kernel engine to autograd: backward = the engine's training reverse pass."""

    @staticmethod
    def forward(ctx, model, eng_out, names, keys, *tensors):
        # everything backward needs is captured HERE: another forward (a validation pass, a second batch of
        # the same loss) before backward() must not change which batch / engine this node differentiates
        ctx.model, ctx.eng_out, ctx.names, ctx.keys = model, eng_out, names, keys
        ctx.engine = model._get_engine()
        ctx.atoms_per_graph = list(eng_out.extras["train_state"]["b"].atoms_per_graph)
        ctx.is_intensive = bool(model.is_intensive)
        return tuple(t.clone() for t in tensors[: len(keys)])

    @staticmethod
    def backward(ctx, *g_outs):
        out = ctx.eng_out
        if "train_state" not in out.extras:
            raise RuntimeError(
                "chgnet_b200: backward through this CHGNet.forward output ran twice; the saved activations are "
                "released by the first backward (retain_graph is not supported) - call forward again")
        g = {k: v.contiguous() for k, v in zip(ctx.keys, g_outs)}
        n = torch.tensor(ctx.atoms_per_graph, device=g["e"].device, dtype=g["e"].dtype)
        seed_e = g["e"] / n if ctx.is_intensive else g["e"]  # d/d(extensive model energy)
        G = ctx.engine.param_grads(out, seed_e.contiguous(), g.get("m"), g.get("f"), g.get("s"))
        grads = unpack_grads(G, ctx.model.state_dict())
        return (None, None, None, None, *[None] * len(ctx.keys), *[grads[k] for k in ctx.names])


class _Node(nn.Module):
    """Plain container used to reproduce the reference's dotted parameter names."""


class GraphConverter:
    """Structure -> CrystalGraph on the host (stand-in for the reference's
    ``CrystalGraphConverter``, reference chgnet/graph/converter.py:102-190; the
    GPU builder is row f1 of SURVEY.md §8).  Accepts any object with
    ``frac_coords``, ``lattice.matrix`` and ``atomic_numbers`` (pymatgen
    ``Structure`` qualifies) or a ``(atomic_numbers, frac_coords, lattice)`` tuple."""

    def __init__(self, atom_graph_cutoff: float = 6, bond_graph_cutoff: float = 3, *,
                 on_isolated_atoms: str = "error", **_: Any) -> None:
        if on_isolated_atoms not in ("ignore", "warn", "error"):
            raise ValueError(f"{on_isolated_atoms=} must be 'ignore', 'warn' or 'error'")
        self.atom_graph_cutoff = atom_graph_cutoff
        self.bond_graph_cutoff = atom_graph_cutoff if bond_graph_cutoff is None else bond_graph_cutoff
        self.on_isolated_atoms = on_isolated_atoms  # reference converter.py:42, 160-174

    def __call__(self, structure, graph_id=None, mp_id=None) -> CrystalGraph:
        from chgnet_b200 import graphgen

        if isinstance(structure, tuple):
            z, frac, lat = structure
        else:
            z = getattr(structure, "atomic_numbers", None)
            if z is None:
                z = [site.specie.Z for site in structure]
            frac = structure.frac_coords
            lat = structure.lattice.matrix if hasattr(structure.lattice, "matrix") else structure.lattice
        g = graphgen.make_crystal_graph(
            np.asarray(z), np.asarray(frac), np.asarray(lat), atom_graph_cutoff=self.atom_graph_cutoff,
            bond_graph_cutoff=self.bond_graph_cutoff, graph_id=graph_id)
        g.mp_id = mp_id
        if self.on_isolated_atoms != "ignore":
            n_atoms = len(g.atomic_number)
            centers = g.atom_graph[:, 0] if g.atom_graph.dim() == 2 and len(g.atom_graph) else torch.zeros(0, dtype=torch.int64)
            n_isolated_atoms = n_atoms - int(torch.unique(centers).numel())
            if n_isolated_atoms:
                atom_graph_cutoff = self.atom_graph_cutoff
                msg = (f"Structure {graph_id=} has {n_isolated_atoms} isolated atom(s) with "
                       f"{atom_graph_cutoff=}. CHGNet calculation will likely go wrong")
                if self.on_isolated_atoms == "error":
                    raise ValueError(msg)
                import sys

                print(msg, file=sys.stderr)
        return g

    def convert_many(self, structures, n_threads: int | None = None) -> list[CrystalGraph]:
        """Graphs of many structures, built concurrently: the native builder (csrc/graph_builder.cu, entered through
        ctypes, which releases the GIL) runs on a thread pool, one structure per task.  Same graphs, same order and the
        same isolated-atom handling as calling the converter in a loop (what the reference's ``predict_structure`` does,
        model.py:578-583)."""
        structures = list(structures)
        if n_threads is None:
            n_threads = min(16, os.cpu_count() or 1)
        if n_threads <= 1 or len(structures) < 4:
            return [self(s) for s in structures]
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=min(n_threads, len(structures))) as ex:
            return list(ex.map(self, structures))

    def __repr__(self) -> str:
        return (f"GraphConverter(atom_graph_cutoff={self.atom_graph_cutoff}, "
                f"bond_graph_cutoff={self.bond_graph_cutoff})")


class StaticGraphEvaluator:
    """``predict_graph`` for a fixed list of graphs evaluated many times with updated coordinates.

    The batch descriptor (indices, CSR structures) is built once and stays on the device; ``update`` overwrites the
    fractional coordinates and / or lattices in place; ``__call__`` launches ONE captured CUDA graph of ``chg_forward``
    (native.NativeForward.replay) instead of ~130 kernels - a 8-atom cell goes from 1.2 ms to a fraction of that.  The
    neighbour lists are NOT rebuilt: the caller guarantees that no pair crosses a cutoff (pairs beyond the cutoffs have
    zero weight, so slightly too LARGE lists are harmless; build the graphs with a larger cutoff for a margin).
    Outputs: the same dicts as ``predict_graph`` (reference model.py:593-665)."""

    def __init__(self, model: "CHGNet", graph, task: str = "efsm") -> None:
        valid_tasks = get_args(PredTask)
        if task not in valid_tasks:
            raise ValueError(f"Invalid {task=}. Must be one of {valid_tasks}.")
        self.model, self.task = model, task
        self.single = is_graph_like(graph)
        graphs = [graph] if self.single else list(graph)
        model.eval()
        need_grad = "f" in task or "s" in task
        self.batch = build_batch(graphs, model.device, with_reverse=need_grad,
                                 compact_bonds=not model._arch.get("mlp_out_bias", False))
        self._bounds = np.cumsum(self.batch.atoms_per_graph)[:-1]

    def update(self, frac=None, lattice=None) -> None:
        """New fractional coordinates ``[N_total, 3]`` (atoms of all graphs, in order) and / or lattices ``[B, 3, 3]``."""
        b = self.batch
        if frac is not None:
            b.frac.copy_(torch.as_tensor(np.asarray(frac, dtype=np.float32)).reshape(b.n_atoms, 3), non_blocking=True)
        if lattice is not None:
            lat = torch.as_tensor(np.asarray(lattice, dtype=np.float32)).reshape(b.n_graphs, 9).to(b.lattice.device)
            b.lattice.copy_(lat)
            cell = b.lattice.view(-1, 3, 3)
            b.volume.copy_((cell[:, 0] * torch.linalg.cross(cell[:, 1], cell[:, 2])).sum(dim=1))

    def __call__(self, return_site_energies: bool = False):
        m = self.model
        raw = m._run(None, self.task, return_site_energies, False, False, batch=self.batch, replay=True)
        n = self.batch.n_graphs
        preds: list[dict[str, np.ndarray]] = [{} for _ in range(n)]
        for key in ("e", "f", "s", "m", "site_energies"):
            if key not in raw:
                continue
            host = raw[key].cpu().numpy()
            parts = np.split(host, self._bounds) if key in m._PER_ATOM else [host[i] for i in range(n)]
            for i, part in enumerate(parts):
                preds[i][key] = np.asarray(part)
        return preds[0] if self.single else preds


class CHGNet(nn.Module):
    """Crystal Hamiltonian Graph neural Network — B200 kernel path."""

    def __init__(
        self,
        *,
        atom_fea_dim: int = 64,
        bond_fea_dim: int = 64,
        angle_fea_dim: int = 64,
        composition_model: str | nn.Module | None = "MPtrj",
        num_radial: int = 31,
        num_angular: int = 31,
        n_conv: int = 4,
        atom_conv_hidden_dim: Sequence[int] | int = 64,
        update_bond: bool = True,
        bond_conv_hidden_dim: Sequence[int] | int = 64,
        update_angle: bool = True,
        angle_layer_hidden_dim: Sequence[int] | int = 0,
        conv_dropout: float = 0,
        read_out: str = "ave",
        mlp_hidden_dims: Sequence[int] | int = (64, 64, 64),
        mlp_dropout: float = 0,
        mlp_first: bool = True,
        is_intensive: bool = True,
        non_linearity: str = "silu",
        atom_graph_cutoff: float = 6,
        bond_graph_cutoff: float = 3,
        graph_converter_algorithm: str = "fast",
        cutoff_coeff: int = 8,
        learnable_rbf: bool = True,
        gMLP_norm: str | None = "layer",  # noqa: N803
        readout_norm: str | None = "layer",
        version: str | None = None,
        **kwargs,
    ) -> None:
        self.model_args = {k: v for k, v in locals().items() if k not in {"self", "__class__", "kwargs"}}
        self.model_args.update(kwargs)
        if version:
            self.model_args["version"] = version
        super().__init__()
        if isinstance(composition_model, nn.Module):
            raise NotImplementedError("custom composition_model modules are not supported; pass a table name or None")
        if non_linearity != "silu":
            raise NotImplementedError("chgnet_b200 kernels implement non_linearity='silu' only")
        if not mlp_first:
            raise NotImplementedError("chgnet_b200 kernels implement mlp_first=True (per-site energies) only")
        if conv_dropout or mlp_dropout:
            raise NotImplementedError("dropout is not implemented (all pretrained models use 0)")
        self.atom_fea_dim, self.bond_fea_dim = atom_fea_dim, bond_fea_dim
        self.is_intensive, self.n_conv, self.mlp_first = is_intensive, n_conv, mlp_first
        a = dict(self.model_args)
        a["conv_norm"] = kwargs.get("conv_norm")
        a["mlp_out_bias"] = kwargs.get("mlp_out_bias", False)
        self._arch = a
        self.graph_converter = GraphConverter(atom_graph_cutoff, bond_graph_cutoff)
        frozen = {"composition_model.fc.weight"}
        if not learnable_rbf:
            frozen |= {"bond_basis_expansion.rbf_expansion_ag.frequencies",
                       "bond_basis_expansion.rbf_expansion_bg.frequencies",
                       "angle_basis_expansion.fourier_expansion.frequencies"}
        for name, (shape, kind) in _param_specs(a).items():
            self._register(name, _init_param(shape, kind, a), trainable=name not in frozen,
                           as_buffer=(not learnable_rbf and name.endswith("frequencies")))
        self._engine: Engine | None = None
        self._engine_key: tuple | None = None
        self._native = None  # native.NativeForward (inference)
        self._native_key: tuple | None = None
        self.last_batch: DeviceBatch | None = None
        version_str = f" v{version}" if version else ""
        print(f"CHGNet{version_str} initialized with {self.n_params:,} parameters")

    # ------------------------------------------------------------------ plumbing
    def _register(self, dotted: str, value: Tensor, *, trainable: bool, as_buffer: bool = False) -> None:
        *path, leaf = dotted.split(".")
        mod: nn.Module = self
        for part in path:
            if part not in mod._modules:
                mod.add_module(part, _Node())
            mod = mod._modules[part]
        if as_buffer:
            mod.register_buffer(leaf, value)
        else:
            mod.register_parameter(leaf, nn.Parameter(value, requires_grad=trainable))

    @property
    def version(self) -> str | None:
        return self.model_args.get("version")

    @property
    def n_params(self) -> int:
        return sum(p.numel() for p in self.parameters())

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def _get_engine_checks(self) -> None:
        a = self._arch
        for name in ("atom_conv_hidden_dim", "bond_conv_hidden_dim"):
            if a[name] != 64 and list(np.atleast_1d(a[name])) != [64]:
                raise NotImplementedError(f"{name} must be 64 for the CUDA kernels")
        if a["angle_layer_hidden_dim"] not in (0, None):
            raise NotImplementedError("angle_layer_hidden_dim must be 0 for the CUDA kernels")
        if a["conv_norm"] is not None:
            raise NotImplementedError("conv_norm is not supported by the CUDA kernels")

    def _get_engine(self) -> Engine:
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError(
                "chgnet_b200.CHGNet has no CPU path: move the model to a CUDA device (B200) first "
                f"(parameters are on {dev})")
        sd = self.state_dict()
        key = (str(dev), tuple(int(v._version) for v in sd.values()), tuple(v.data_ptr() for v in sd.values()))
        if self._engine is None or key != self._engine_key:
            from chgnet_b200._lib import CudaKernels

            self._get_engine_checks()
            pw = pack_weights(sd, self.model_args, device=dev)
            self._engine = Engine(pw, CudaKernels(dev))
            self._engine_key = key
        return self._engine

    def _get_native(self):
        """Inference path: packed weights on the device + ONE ``chg_forward`` call per batch (native.py)."""
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError(
                "chgnet_b200.CHGNet has no CPU path: move the model to a CUDA device (B200) first "
                f"(parameters are on {dev})")
        sd = self.state_dict()
        key = (str(dev), tuple(int(v._version) for v in sd.values()), tuple(v.data_ptr() for v in sd.values()))
        if self._native is None or key != self._native_key:
            from chgnet_b200.native import NativeForward

            self._get_engine_checks()
            self._native = NativeForward(sd, self.model_args, dev)
            self._native_key = key
        return self._native

    def _engine_cache_key(self) -> tuple:
        sd = self.state_dict()
        return (str(self.device), tuple(int(v._version) for v in sd.values()), tuple(v.data_ptr() for v in sd.values()))

    def _mark_engine_current(self) -> None:
        """The training engine's packed weights were refreshed in place (Trainer.refresh_packed_weights): keep the
        Engine object, record that it matches the parameters as they are now."""
        if self._engine is not None:
            self._engine_key = self._engine_cache_key()

    def mark_params_updated(self) -> None:
        """Call after changing parameter storage in place from outside autograd (e.g. the fused Adam
        kernel): the packed kernel weights are rebuilt on the next forward."""
        self._engine_key = None
        self._native_key = None

    # ------------------------------------------------------------------ forward
    def _run(self, graphs, task, return_site_energies, return_atom_feas, return_crystal_feas,
             train: bool = False, batch: DeviceBatch | None = None, replay: bool = False) -> dict[str, Any]:
        """One batch through the kernels; returns BATCHED device tensors.

        Inference = one native ``chg_forward`` call (native.py; ``CHGNET_B200_ENGINE=python`` selects the
        call-by-call Python schedule of engine.py instead, same kernels); training = engine.py."""
        need_grad = "f" in task or "s" in task
        # mlp_out bias (0.2.0) touches every bond: no bond-graph compaction in that case
        compact = not self._arch.get("mlp_out_bias", False)
        if batch is None:
            batch = build_batch(graphs, self.device, with_reverse=need_grad or train, compact_bonds=compact)
        self.last_batch = batch
        if not train and os.environ.get("CHGNET_B200_ENGINE", "native") != "python":
            nat = self._get_native()
            if replay and not return_crystal_feas:  # same resident batch again: one CUDA-graph launch (native.py)
                res = nat.replay(batch, need_grad=need_grad, need_magmom="m" in task, need_atom_fea=return_atom_feas)
            else:
                res = nat(batch, need_grad=need_grad, need_magmom="m" in task, need_atom_fea=return_atom_feas,
                          need_crystal_fea=return_crystal_feas)
            from chgnet_b200.engine import EngineOutput

            out = EngineOutput(energy=res["energy"], e_ref=res["e_ref"], site_e=res["site_e"], magmom=res.get("magmom"),
                               atom_fea=res.get("atom_fea"), crystal_fea=res.get("crystal_fea"), force=res.get("force"),
                               virial=res.get("virial"))
            atom_ref = nat.atom_ref
        else:
            engine = self._get_engine()
            out = engine.run(batch, need_grad=need_grad, need_magmom="m" in task, need_atom_fea=return_atom_feas,
                             need_crystal_fea=return_crystal_feas, train=train)
            if train and need_grad:  # force pass; keeps the adjoints the second-order pass needs
                engine.input_grads(out, record=True)
            atom_ref = engine.pw.atom_ref
        self._last_out = out
        n_dev = torch.tensor(batch.atoms_per_graph, device=self.device)
        raw: dict[str, Any] = {"atoms_per_graph": n_dev}
        if return_atom_feas:
            raw["atom_fea"] = out.atom_fea
        if "m" in task:
            raw["m"] = out.magmom
        if return_site_energies:
            raw["site_energies"] = out.site_e + atom_ref[batch.z.long() - 1]
        if return_crystal_feas:
            raw["crystal_fea"] = out.crystal_fea
        if "f" in task:
            raw["f"] = out.force.to(torch.float32)
        if "s" in task:
            scale = EV_A3_TO_GPA / batch.volume.to(torch.float64)
            raw["s"] = (out.virial.view(-1, 3, 3) * scale[:, None, None]).to(torch.float32)
        total = out.energy + out.e_ref
        if self.is_intensive:
            total = total / n_dev
        raw["e"] = total.to(torch.float32)
        return raw

    _PER_ATOM = ("atom_fea", "m", "site_energies", "f")

    def forward(
        self,
        graphs: Sequence[CrystalGraph],
        *,
        task: PredTask = "e",
        return_site_energies: bool = False,
        return_atom_feas: bool = False,
        return_crystal_feas: bool = False,
    ) -> dict[str, Tensor]:
        """Prediction for a list of CrystalGraphs (reference model.py:330-387): ``e`` Tensor[B],
        ``f`` / ``m`` / ``site_energies`` / ``atom_fea`` lists of per-graph tensors, ``s`` list of
        [3,3], ``crystal_fea`` Tensor[B,64], ``atoms_per_graph``."""
        train = self.training and torch.is_grad_enabled()
        raw = self._run(graphs, task, return_site_energies, return_atom_feas, return_crystal_feas, train=train)
        if train:
            # every output carries autograd history to the parameters (the reference's training mode,
            # model.py:518-535 create_graph=True / trainer.py:398-410): backward() runs the engine's
            # training reverse pass, with the second-order pass when f / s received a gradient
            names = [n for n, p in self.named_parameters() if p.requires_grad]
            params = [p for _, p in self.named_parameters() if p.requires_grad]
            keys = [k for k in ("e", "m", "f", "s") if raw.get(k) is not None]
            outs = _ParamGradBridge.apply(self, self._last_out, names, keys, *[raw[k] for k in keys], *params)
            for k, v in zip(keys, outs):
                raw[k] = v
        n_list = self.last_batch.atoms_per_graph
        pred: dict[str, Any] = {}
        for key, val in raw.items():
            if key in self._PER_ATOM:
                parts = torch.split(val, n_list)
                pred[key] = parts if key == "atom_fea" else list(parts)
            elif key == "s":
                pred[key] = list(val.unbind(0))
            else:
                pred[key] = val
        return pred

    # ------------------------------------------------------------------ predict API
    def predict_structure(self, structure, *, task: PredTask = "efsm", return_site_energies: bool = False,
                          return_atom_feas: bool = False, return_crystal_feas: bool = False, batch_size: int = 16):
        """Predict from structure(s) (reference model.py:544-591)."""
        if self.graph_converter is None:
            raise ValueError("graph_converter cannot be None!")
        single = hasattr(structure, "frac_coords") or isinstance(structure, tuple)
        if (single and isinstance(self.graph_converter, GraphConverter) and self.device.type == "cuda"
                and os.environ.get("CHGNET_B200_GRAPH", "device") == "device"):
            return self._predict_structure_device(structure, task, return_site_energies, return_atom_feas, return_crystal_feas)
        structures = [structure] if single else structure
        if (not single and isinstance(self.graph_converter, GraphConverter)
                and os.environ.get("CHGNET_B200_GRAPH", "device") != "python"):
            return self._predict_structures_native(list(structures), task, return_site_energies, return_atom_feas,
                                                   return_crystal_feas, batch_size)
        convert_many = getattr(self.graph_converter, "convert_many", None)
        graphs = convert_many(structures) if convert_many is not None else [self.graph_converter(s) for s in structures]
        return self.predict_graph(graphs[0] if single else graphs, task=task,
                                  return_site_energies=return_site_energies, return_atom_feas=return_atom_feas,
                                  return_crystal_feas=return_crystal_feas, batch_size=batch_size)

    @staticmethod
    def _structure_arrays(structure):
        if isinstance(structure, tuple):
            z, frac, lat = structure
        else:
            z = getattr(structure, "atomic_numbers", None)
            if z is None:
                z = [site.specie.Z for site in structure]
            frac = structure.frac_coords
            lat = structure.lattice.matrix if hasattr(structure.lattice, "matrix") else structure.lattice
        return (np.ascontiguousarray(z, dtype=np.int32).reshape(-1), np.ascontiguousarray(frac, dtype=np.float64).reshape(-1, 3),
                np.ascontiguousarray(lat, dtype=np.float64).reshape(3, 3))

    def structures_to_batch(self, structures, *, with_reverse: bool = True):
        """``list[structure] -> DeviceBatch`` without per-structure Python objects: the graphs are built concurrently by
        the library's worker threads (``chg_graph_build_many``) and packed straight out of the builder's memory
        (``chg_graph_views`` -> ``chg_pack_batch_wire``).  Identical to converting every structure with the
        ``GraphConverter`` and batching the CrystalGraphs (tests/test_graph_builder.py)."""
        import ctypes

        from chgnet_b200._lib import ChgnetB200Error, load_library
        from chgnet_b200.batch import build_batch

        lib = load_library()
        if not getattr(lib, "_graph_many_bound", False):
            vp = ctypes.c_void_p
            lib.chg_graph_build_many.restype = ctypes.c_int32
            lib.chg_graph_build_many.argtypes = [ctypes.c_int32, vp, vp, vp, ctypes.c_double, ctypes.c_double, vp]
            lib.chg_graph_views.restype = ctypes.c_int32
            lib.chg_graph_views.argtypes = [ctypes.c_int32, vp, vp, vp, vp]
            lib.chg_graph_free_many.restype = None
            lib.chg_graph_free_many.argtypes = [ctypes.c_int32, vp]
            lib._graph_many_bound = True
        gc = self.graph_converter
        arrays = [self._structure_arrays(s) for s in structures]
        n = len(arrays)
        n_at = np.array([len(a[0]) for a in arrays], dtype=np.int32)
        frac_p = np.array([a[1].ctypes.data for a in arrays], dtype=np.uint64)
        lat_p = np.array([a[2].ctypes.data for a in arrays], dtype=np.uint64)
        handles = np.zeros(max(n, 1), dtype=np.uint64)
        rc = lib.chg_graph_build_many(n, frac_p.ctypes.data, lat_p.ctypes.data, n_at.ctypes.data, float(gc.atom_graph_cutoff),
                                      float(gc.bond_graph_cutoff), handles.ctypes.data)
        try:
            if rc != 0:
                msg = lib.chg_last_error().decode()
                raise (ValueError if "not complete" in msg else ChgnetB200Error)(msg)
            counts3, ptrs5 = np.empty((n, 3), dtype=np.int64), np.empty((n, 5), dtype=np.uint64)
            n_iso = np.zeros(max(n, 1), dtype=np.int32)
            lib.chg_graph_views(n, handles.ctypes.data, counts3.ctypes.data, ptrs5.ctypes.data, n_iso.ctypes.data)
            if gc.on_isolated_atoms != "ignore" and n_iso.any():
                for i in np.nonzero(n_iso)[0]:
                    n_isolated_atoms, atom_graph_cutoff, graph_id = int(n_iso[i]), gc.atom_graph_cutoff, None
                    msg = (f"Structure {graph_id=} has {n_isolated_atoms} isolated atom(s) with "
                           f"{atom_graph_cutoff=}. CHGNet calculation will likely go wrong")
                    if gc.on_isolated_atoms == "error":
                        raise ValueError(msg)
                    import sys

                    print(msg, file=sys.stderr)
            # fp32 / int32 copies of the per-atom and per-structure inputs, one array each, addressed by offsets
            z_all = np.concatenate([a[0] for a in arrays]) if n else np.zeros(0, np.int32)
            frac_all = np.concatenate([a[1] for a in arrays]).astype(np.float32) if n else np.zeros((0, 3), np.float32)
            lat_all = np.stack([a[2] for a in arrays]).astype(np.float32).reshape(n, 9) if n else np.zeros((0, 9), np.float32)
            a_off = np.concatenate([[0], np.cumsum(n_at[:-1], dtype=np.int64)]).astype(np.uint64) if n else np.zeros(0, np.uint64)
            counts = np.empty((n, 4), dtype=np.int64)
            counts[:, 0], counts[:, 1:] = n_at, counts3
            ptrs = np.empty((n, 8), dtype=np.uint64)
            ptrs[:, 0] = np.uint64(z_all.ctypes.data) + a_off * np.uint64(4)
            ptrs[:, 1] = np.uint64(frac_all.ctypes.data) + a_off * np.uint64(12)
            for k in range(5):
                ptrs[:, 2 + k] = ptrs5[:, k]
            ptrs[:, 7] = np.uint64(lat_all.ctypes.data) + np.arange(n, dtype=np.uint64) * np.uint64(36)
            # both packers copy into their staging buffers before they return: the handles can be freed right after
            return build_batch(None, self.device, with_reverse=with_reverse,
                               compact_bonds=not self._arch.get("mlp_out_bias", False), packed=(counts, ptrs))
        finally:
            lib.chg_graph_free_many(n, handles.ctypes.data)

    def _predict_structures_native(self, structures, task, return_site_energies, return_atom_feas, return_crystal_feas,
                                   batch_size):
        """``predict_structure`` of a list: chunks of ``batch_size`` structures through ``structures_to_batch``; same
        graphs, chunking and outputs as converting every structure and calling ``predict_graph`` (reference
        model.py:544-591)."""
        valid_tasks = get_args(PredTask)
        if task not in valid_tasks:
            raise ValueError(f"Invalid {task=}. Must be one of {valid_tasks}.")
        self.eval()
        need_grad = "f" in task or "s" in task
        predictions: list[dict[str, np.ndarray]] = [{} for _ in structures]
        for start in range(0, len(structures), batch_size):
            batch = self.structures_to_batch(structures[start : start + batch_size], with_reverse=need_grad)
            n = batch.n_graphs
            raw = self._run(None, task, return_site_energies, return_atom_feas, return_crystal_feas, batch=batch)
            bounds = np.cumsum(batch.atoms_per_graph)[:-1]
            for key in ("e", "f", "s", "m", "site_energies", "atom_fea", "crystal_fea"):
                if key not in raw:
                    continue
                host = raw[key].cpu().numpy()
                parts = np.split(host, bounds) if key in self._PER_ATOM else [host[i] for i in range(n)]
                for i, part in enumerate(parts):
                    predictions[start + i][key] = np.asarray(part)
        return predictions

    def _predict_structure_device(self, structure, task, return_site_energies, return_atom_feas, return_crystal_feas):
        """One structure, graph built ON THE DEVICE (chgnet_b200.graph_device: the same edges / angles as the host
        converter, bit for bit): only the atomic numbers, fractional coordinates and the lattice cross PCIe."""
        from chgnet_b200.graph_device import DeviceGraphBuilder

        valid_tasks = get_args(PredTask)
        if task not in valid_tasks:
            raise ValueError(f"Invalid {task=}. Must be one of {valid_tasks}.")
        if isinstance(structure, tuple):
            z, frac, lat = structure
        else:
            z = getattr(structure, "atomic_numbers", None)
            if z is None:
                z = [site.specie.Z for site in structure]
            frac = structure.frac_coords
            lat = structure.lattice.matrix if hasattr(structure.lattice, "matrix") else structure.lattice
        gc = self.graph_converter
        key = (str(self.device), float(gc.atom_graph_cutoff), float(gc.bond_graph_cutoff))
        if getattr(self, "_dev_builder_key", None) != key:
            self._dev_builder = DeviceGraphBuilder(self.device, gc.atom_graph_cutoff, gc.bond_graph_cutoff)
            self._dev_builder_key = key
        self.eval()
        need_grad = "f" in task or "s" in task
        f64 = torch.as_tensor(np.ascontiguousarray(np.asarray(frac, dtype=np.float64).reshape(-1, 3))).to(self.device)
        batch = self._dev_builder.build_batch(np.asarray(z), f64, np.asarray(lat, dtype=np.float64), with_reverse=need_grad,
                                              compact_bonds=not self._arch.get("mlp_out_bias", False))
        if gc.on_isolated_atoms != "ignore" and batch.n_atoms:
            n_isolated_atoms = int((batch.ptr_c[1:] == batch.ptr_c[:-1]).sum().item())
            if n_isolated_atoms:
                atom_graph_cutoff, graph_id = gc.atom_graph_cutoff, None
                msg = (f"Structure {graph_id=} has {n_isolated_atoms} isolated atom(s) with "
                       f"{atom_graph_cutoff=}. CHGNet calculation will likely go wrong")
                if gc.on_isolated_atoms == "error":
                    raise ValueError(msg)
                import sys

                print(msg, file=sys.stderr)
        raw = self._run(None, task, return_site_energies, return_atom_feas, return_crystal_feas, batch=batch)
        out: dict[str, np.ndarray] = {}
        for key_ in ("e", "f", "s", "m", "site_energies", "atom_fea", "crystal_fea"):
            if key_ in raw:
                host = raw[key_].cpu().numpy()
                out[key_] = np.asarray(host if key_ in self._PER_ATOM else host[0])
        return out

    def predict_graph(self, graph, *, task: PredTask = "efsm", return_site_energies: bool = False,
                      return_atom_feas: bool = False, return_crystal_feas: bool = False, batch_size: int = 16):
        """Predict from CrystalGraph(s); numpy outputs (reference model.py:593-665)."""
        if not (is_graph_like(graph) or isinstance(graph, Sequence)):
            raise TypeError(f"{type(graph)=} must be CrystalGraph or list of CrystalGraphs")
        valid_tasks = get_args(PredTask)
        if task not in valid_tasks:
            raise ValueError(f"Invalid {task=}. Must be one of {valid_tasks}.")
        single = is_graph_like(graph)
        graphs = [graph] if single else list(graph)
        self.eval()
        predictions: list[dict[str, np.ndarray]] = [{} for _ in graphs]
        for start in range(0, len(graphs), batch_size):
            chunk = graphs[start : start + batch_size]
            raw = self._run(chunk, task, return_site_energies, return_atom_feas, return_crystal_feas)
            bounds = np.cumsum(self.last_batch.atoms_per_graph)[:-1]
            for key in ("e", "f", "s", "m", "site_energies", "atom_fea", "crystal_fea"):
                if key not in raw:
                    continue
                host = raw[key].cpu().numpy()  # ONE device->host copy per key, split on the host
                parts = np.split(host, bounds) if key in self._PER_ATOM else [host[i] for i in range(len(chunk))]
                for i, part in enumerate(parts):
                    predictions[start + i][key] = np.asarray(part)
        return predictions[0] if single else predictions

    def static_evaluator(self, graph, *, task: PredTask = "efsm"):
        """Evaluator for graph(s) whose TOPOLOGY stays fixed while coordinates / cells change (finite differences,
        phonon displacements, line searches): see ``StaticGraphEvaluator``."""
        return StaticGraphEvaluator(self, graph, task)

    # ------------------------------------------------------------------ (de)serialisation
    def as_dict(self) -> dict:
        return {"state_dict": self.state_dict(), "model_args": self.model_args}

    def todict(self) -> dict:
        return {"model_name": type(self).__name__, "model_args": self.model_args}

    @classmethod
    def from_dict(cls, dct: dict, **kwargs):
        model = cls(**dct["model_args"], **kwargs)
        model.load_state_dict(dct["state_dict"])
        return model

    @classmethod
    def from_file(cls, path: str, **kwargs):
        if path.endswith(".npz"):  # plain-array export of a state_dict (tests/golden), optionally with its model_args
            import json

            with np.load(path) as f:
                sd = {k: torch.from_numpy(f[k]) for k in f.files if k != "__model_args__"}
                args = json.loads(str(f["__model_args__"])) if "__model_args__" in f.files else {}
            args.update(kwargs)
            return cls.from_dict({"model_args": args, "state_dict": sd})
        state = torch.load(path, map_location=torch.device("cpu"), weights_only=False)
        return cls.from_dict(state["model"], **kwargs)

    @classmethod
    def load(cls, *, model_name: str = "0.3.0", use_device: str | None = None, check_cuda_mem: bool = False,
             verbose: bool = True):
        """Load a pretrained model (reference model.py:690-745).  Checkpoints are looked up in
        $CHGNET_PRETRAINED_DIR, an installed ``chgnet`` package, then the plain-array exports
        under tests/golden."""
        rel = _CHECKPOINTS.get(model_name)
        if rel is None:
            raise ValueError(f"Unknown {model_name=}")
        roots = [os.environ.get("CHGNET_PRETRAINED_DIR")]
        try:
            import importlib.util

            spec = importlib.util.find_spec("chgnet")
            if spec is not None and spec.submodule_search_locations:
                roots.append(os.path.join(list(spec.submodule_search_locations)[0], "pretrained"))
        except (ImportError, ValueError):
            pass
        model = None
        for root in roots:
            if root and os.path.exists(os.path.join(root, rel)):
                model = cls.from_file(os.path.join(root, rel), mlp_out_bias=model_name == "0.2.0", version=model_name)
                break
        if model is None:
            npz = os.path.join(_REPO, "tests", "golden", f"chgnet_{model_name}_weights.npz")
            if not os.path.exists(npz):
                raise FileNotFoundError(f"no checkpoint for {model_name=}; set CHGNET_PRETRAINED_DIR")
            model = cls.from_file(npz, version=model_name, **({"mlp_out_bias": True} if model_name == "0.2.0" else {}))
        device = use_device or os.environ.get("CHGNET_DEVICE") or "cuda"
        if not str(device).startswith("cuda"):
            raise RuntimeError(f"chgnet_b200 runs on CUDA devices only (requested {device!r})")
        model = model.to(device)
        if verbose:
            print(f"CHGNet will run on {device}")
        return model
