"""ctypes binding of ``libchgnet_b200.so`` (the C ABI in include/chgnet_b200.h).

PyTorch is plumbing here: tensors only provide device memory (``data_ptr()``) and
the current CUDA stream.  There is NO fallback: if the shared library is missing
or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_int64, c_void_p

import torch
from torch import Tensor

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libchgnet_b200.so")

P, I, F, I64 = c_void_p, c_int32, c_float, c_int64

# name -> argument ctypes (the trailing stream pointer included); mirrors the header 1:1
SIGNATURES: dict[str, list] = {
    "chg_embed_atoms": [P, P, I, P, P],
    "chg_edge_geometry": [P, P, P, P, P, P, I, P, P, P, P],
    "chg_bond_basis_embed": [P, P, I, P, P, I, F, F, I, P, P, P, P, P, P],
    "chg_bond_basis_bwd": [P, P, I, P, P, I, F, F, I, P, P, P, P, P, P, P],
    "chg_angle_basis_embed": [P, P, P, I, P, I, P, P, P, P],
    "chg_angle_basis_bwd": [P, P, P, I, P, I, P, P, P, P, P],
    "chg_linear": [P, P, I, I, P, P, P, P, I, P, P],
    "chg_gather_rows": [P, P, I, I, P, P],
    "chg_scatter_rows": [P, P, I, I, P, P],
    "chg_atom_conv_fwd": [P, P, P, P, P, P, I, P, P, P, P, P, P, P],
    "chg_atom_conv_bwd": [P, P, P, P, P, P, I, P, P, P, P, P, P, P, P, P],
    "chg_segment_sum": [P, I, P, P, I, I, I, P, I, P],
    "chg_atom_conv_fused": [P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, P],
    "chg_bond_conv_fused": [P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, P, P],
    "chg_bond_conv_fwd": [P, P, P, P, P, P, P, I, P, P, P, P, P, P, P],
    "chg_bond_conv_bwd": [P, P, P, P, P, I, P, P, P, P, P, P, P, P, P],
    "chg_angle_update_fwd": [P, P, P, P, P, P, P, I, P, P, P, P],
    "chg_angle_update_bwd": [P, P, I, P, P, P, P],
    "chg_readout": [P, P, P, I, P, P, P, P, I, P, F, P, P, P, P, P, P, P],
    "chg_magmom": [P, I, P, F, P, P],
    "chg_force_virial": [P, P, P, P, P, P, P, P, P, P, I, P, P, P],
    # Berendsen NVT / NPT with the cell on the device (dynamics_device.DeviceMD)
    "chg_md_partial_blocks": [I],
    "chg_md_cell_step": [P, P, P, I, P, P, I, P],
    "chg_md_kick_drift_cell": [P, P, P, P, I, ctypes.c_double, P, P, P, P, P, I, P],
    "chg_md_kick_partials": [P, P, P, I, ctypes.c_double, P, P],
    # training
    "chg_wgrad": [P, P, I, P, I, P, I, P, I, I, P, I, P, P, P],
    "chg_colsum": [P, I, P, I, P, I, I, P, P],
    "chg_readout_bwd": [P, I, P, P, P, P, I, P, P, P, P, P, P, P, P],
    "chg_magmom_bwd": [P, I, P, F, P, P, P, P],
    "chg_loss_terms": [P, P, I, I, F, P, P, P],
    "chg_adam_step": [P, P, P, P, I64, F, F, F, F, F, I, P],
    # second order (force / stress losses)
    "chg_edge_tangent": [P, P, P, P, P, P, P, P, I, P, P, P],
    "chg_bond_basis_tangent": [P, P, P, I, P, P, I, F, F, I, P, P, P, P, P, P],
    "chg_bond_basis_bwd2": [P, P, P, I, P, P, I, F, F, I, P, P, P, P, P, P],
    "chg_angle_basis_tangent": [P, P, P, P, I, P, I, P, P, P, P],
    "chg_angle_basis_bwd2": [P, P, P, P, I, P, I, P, P, P, P],
    "chg_atom_conv_tan": [P, P, P, P, P, P, P, I, P, P, P, P, P, P, P, P],
    "chg_atom_conv_bwd2": [P, P, P, P, P, P, P, P, P, I, P, P, P, P, P, P, P, P, P],
    "chg_bond_conv_tan": [P, P, P, P, P, P, P, P, I, P, P, P, P, P, P, P, P],
    "chg_bond_conv_bwd2": [P, P, P, P, P, P, P, P, P, I, P, P, P, P, P, P, P, P, P, P],
    "chg_angle_update_tan": [P, P, P, P, P, P, P, I, P, P, P, P, P],
    "chg_angle_update_bwd2": [P, P, P, P, I, P, P, P, P],
    "chg_readout_bwd2": [P, P, I, P, P, P, P, I, P, P, P, P, P, P, P, P, P, P, P, P],
}

_lib = None


class ChgnetB200Error(RuntimeError):
    pass


def load_library(path: str | None = None) -> ctypes.CDLL:
    """dlopen the kernel library; raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise ChgnetB200Error(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C chgnet_b200/csrc`). chgnet_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(path)
    lib.chg_last_error.restype = c_char_p
    lib.chg_last_error.argtypes = []
    lib.chg_abi_version.restype = c_int32
    lib.chg_abi_version.argtypes = []
    lib.chg_launch_count.restype = c_int64
    lib.chg_launch_count.argtypes = []
    lib.chg_set_option.restype = c_int32
    lib.chg_set_option.argtypes = [c_char_p, c_int32]
    lib.chg_wgrad_workspace_floats.restype = c_int64
    lib.chg_wgrad_workspace_floats.argtypes = [c_int32]
    lib.chg_gated_fused_workspace_floats.restype = c_int64
    lib.chg_gated_fused_workspace_floats.argtypes = [c_int32]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = c_int32
        fn.argtypes = argtypes
    _lib = lib
    return lib


def _p(t: Tensor | None):
    if t is None:
        return None
    return t.data_ptr()


class CudaKernels:
    """Python face of the C ABI: one method per entry point, tensors in, nothing returned."""

    name = "cuda"

    def __init__(self, device: torch.device | str | int | None = None) -> None:
        """``device``: the CUDA device whose tensors this object will be handed (default: the current one).
        Every launch runs with that device current and on ITS current stream, whatever the process's
        current device is (``CHGNet.load(use_device='cuda:1')`` in a process sitting on cuda:0)."""
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise ChgnetB200Error("chgnet_b200 needs a CUDA device (B200 / sm_100a); none is visible")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise ChgnetB200Error(f"chgnet_b200 kernels run on CUDA devices only (got {dev})")
        self.device_index = torch.cuda.current_device() if dev.index is None else dev.index

    # ------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device_index).cuda_stream

    def _call(self, name: str, *args) -> None:
        if torch.cuda.current_device() != self.device_index:
            with torch.cuda.device(self.device_index):
                return self._call(name, *args)
        rc = getattr(self.lib, name)(*args, self._stream())
        if rc != 0:
            raise ChgnetB200Error(f"{name} failed ({rc}): {self.lib.chg_last_error().decode()}")

    @staticmethod
    def _chk(*tensors: Tensor | None) -> None:
        for t in tensors:
            if t is not None and (not t.is_cuda or not t.is_contiguous()):
                raise ChgnetB200Error("kernel arguments must be contiguous CUDA tensors")

    def set_option(self, name: str, value: int) -> None:
        """The one run-time option (include/chgnet_b200.h): 'ws_min_rows', the row count from which AtomConv /
        BondConv inference calls run the warp-specialised tcgen05 kernels instead of the FFMA kernels (default
        4096; 0 runs them on any graph)."""
        if self.lib.chg_set_option(name.encode(), int(value)) != 0:
            raise ChgnetB200Error(self.lib.chg_last_error().decode())

    @property
    def launches(self) -> int:
        return int(self.lib.chg_launch_count())

    # ------------------------------------------------------------------ kernels
    def embed_atoms(self, z, emb, x):
        self._chk(z, emb, x)
        self._call("chg_embed_atoms", _p(z), _p(emb), z.shape[0], _p(x))

    def edge_geometry(self, frac, lattice, owner, center, nbr, image, rvec, dist, rhat):
        self._chk(frac, lattice, owner, center, nbr, image, rvec, dist, rhat)
        self._call("chg_edge_geometry", _p(frac), _p(lattice), _p(owner), _p(center), _p(nbr), _p(image),
                   center.shape[0], _p(rvec), _p(dist), _p(rhat))

    def bond_basis_embed(self, dist, u2d, freq_ag, freq_bg, rc_ag, rc_bg, p, w3t, e0, wag, wbg, basis_out=None):
        self._chk(dist, u2d, freq_ag, freq_bg, w3t, e0, wag, wbg, basis_out)
        self._call("chg_bond_basis_embed", _p(dist), _p(u2d), u2d.shape[0], _p(freq_ag), _p(freq_bg),
                   freq_ag.shape[0], float(rc_ag), float(rc_bg), int(p), _p(w3t), _p(e0), _p(wag), _p(wbg),
                   _p(basis_out))

    def bond_basis_bwd(self, dist, u2d, freq_ag, freq_bg, rc_ag, rc_bg, p, w3, g_e0, g_wag, g_wbg, g_dist,
                       g_freq=None):
        self._chk(dist, u2d, freq_ag, freq_bg, w3, g_e0, g_wag, g_wbg, g_dist, g_freq)
        self._call("chg_bond_basis_bwd", _p(dist), _p(u2d), u2d.shape[0], _p(freq_ag), _p(freq_bg),
                   freq_ag.shape[0], float(rc_ag), float(rc_bg), int(p), _p(w3), _p(g_e0), _p(g_wag), _p(g_wbg),
                   _p(g_dist), _p(g_freq))

    def angle_basis_embed(self, rhat, ang_di, ang_dj, freq, wt, a0, basis_out=None):
        self._chk(rhat, ang_di, ang_dj, freq, wt, a0, basis_out)
        self._call("chg_angle_basis_embed", _p(rhat), _p(ang_di), _p(ang_dj), ang_di.shape[0], _p(freq),
                   freq.shape[0], _p(wt), _p(a0), _p(basis_out))

    def angle_basis_bwd(self, rhat, ang_di, ang_dj, freq, w, g_a0, g_rhat, g_freq=None):
        self._chk(rhat, ang_di, ang_dj, freq, w, g_a0, g_rhat, g_freq)
        self._call("chg_angle_basis_bwd", _p(rhat), _p(ang_di), _p(ang_dj), ang_di.shape[0], _p(freq),
                   freq.shape[0], _p(w), _p(g_a0), _p(g_rhat), _p(g_freq))

    def linear(self, x, wt, bias, residual, y, x_rows=None, y_rows=None):
        self._chk(x, wt, bias, residual, y, x_rows, y_rows)
        m = x_rows.shape[0] if x_rows is not None else x.shape[0]
        self._call("chg_linear", _p(x), _p(x_rows), m, x.shape[1], _p(wt), _p(bias), _p(residual), _p(y_rows),
                   wt.shape[1], _p(y))

    def gather_rows(self, src, idx, dst):
        self._chk(src, idx, dst)
        self._call("chg_gather_rows", _p(src), _p(idx), idx.shape[0], src.shape[1], _p(dst))

    def scatter_rows(self, src, idx, dst):
        self._chk(src, idx, dst)
        self._call("chg_scatter_rows", _p(src), _p(idx), idx.shape[0], src.shape[1], _p(dst))

    def atom_conv_fwd(self, pcn, pe, wag, center, nbr, d2u, w2t, b2, ln, msg, save_p, save_pre=None):
        self._chk(pcn, pe, wag, center, nbr, d2u, w2t, b2, ln, msg, save_p, save_pre)
        self._call("chg_atom_conv_fwd", _p(pcn), _p(pe), _p(wag), _p(center), _p(nbr), _p(d2u), center.shape[0],
                   _p(w2t), _p(b2), _p(ln), _p(msg), _p(save_p), _p(save_pre))

    def atom_conv_bwd(self, pcn, pe, wag, center, nbr, d2u, save_p, g_agg, w2, ln, g_pre, g_w, g_p=None, g_ln=None):
        self._chk(pcn, pe, wag, center, nbr, d2u, save_p, g_agg, w2, ln, g_pre, g_w, g_p, g_ln)
        self._call("chg_atom_conv_bwd", _p(pcn), _p(pe), _p(wag), _p(center), _p(nbr), _p(d2u), center.shape[0],
                   _p(save_p), _p(g_agg), _p(w2), _p(ln), _p(g_pre), _p(g_w), _p(g_p), _p(g_ln))

    def _fused_work(self, n_rows: int, device) -> Tensor:
        """Grow-only scratch of the fused message + aggregation kernels (strip partials; the message itself
        when a call below 'ws_min_rows' takes the unfused FFMA path)."""
        need = int(self.lib.chg_gated_fused_workspace_floats(int(n_rows)))
        ws = getattr(self, "_fws", None)
        if ws is None or ws.device != device or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.float32, device=device)
            self._fws = ws
        return ws

    def atom_conv_fused(self, pcn, pe, wag, center, nbr, d2u, ptr_c, w2t, b2, ln, agg, save_p):
        self._chk(pcn, pe, wag, center, nbr, d2u, ptr_c, w2t, b2, ln, agg, save_p)
        self._call("chg_atom_conv_fused", _p(pcn), _p(pe), _p(wag), _p(center), _p(nbr), _p(d2u), _p(ptr_c), center.shape[0],
                   agg.shape[0], _p(w2t), _p(b2), _p(ln), _p(agg), _p(save_p), _p(self._fused_work(center.shape[0], agg.device)))

    def bond_conv_fused(self, pij, px, pa, wbg, ang_atom, ang_i, ang_j, ptr_i, w2t, b2, ln, agg, save_pre, save_p):
        self._chk(pij, px, pa, wbg, ang_atom, ang_i, ang_j, ptr_i, w2t, b2, ln, agg, save_pre, save_p)
        self._call("chg_bond_conv_fused", _p(pij), _p(px), _p(pa), _p(wbg), _p(ang_atom), _p(ang_i), _p(ang_j), _p(ptr_i),
                   ang_i.shape[0], agg.shape[0], _p(w2t), _p(b2), _p(ln), _p(agg), _p(save_pre), _p(save_p),
                   _p(self._fused_work(ang_i.shape[0], agg.device)))

    def segment_sum(self, data, perm, ptr, accumulate, out):
        self._chk(data, perm, ptr)
        if not out.is_cuda or out.stride(1) != 1:
            raise ChgnetB200Error("segment_sum output must be a CUDA tensor with unit column stride")
        n_items = data.shape[0] if perm is None else perm.shape[0]
        self._call("chg_segment_sum", _p(data), data.shape[1], _p(perm), _p(ptr), ptr.shape[0] - 1, n_items,
                   int(accumulate), _p(out), out.stride(0))

    def bond_conv_fwd(self, pij, px, pa, wbg, ang_atom, ang_i, ang_j, w2t, b2, ln, upd, save_pre, save_p):
        self._chk(pij, px, pa, wbg, ang_atom, ang_i, ang_j, w2t, b2, ln, upd, save_pre, save_p)
        self._call("chg_bond_conv_fwd", _p(pij), _p(px), _p(pa), _p(wbg), _p(ang_atom), _p(ang_i), _p(ang_j),
                   ang_i.shape[0], _p(w2t), _p(b2), _p(ln), _p(upd), _p(save_pre), _p(save_p))

    def bond_conv_bwd(self, save_pre, save_p, wbg, ang_i, ang_j, g_agg, w2, ln, g_pre, gw_i, gw_j, g_p=None,
                      g_ln=None):
        self._chk(save_pre, save_p, wbg, ang_i, ang_j, g_agg, w2, ln, g_pre, gw_i, gw_j, g_p, g_ln)
        self._call("chg_bond_conv_bwd", _p(save_pre), _p(save_p), _p(wbg), _p(ang_i), _p(ang_j), ang_i.shape[0],
                   _p(g_agg), _p(w2), _p(ln), _p(g_pre), _p(gw_i), _p(gw_j), _p(g_p), _p(g_ln))

    def angle_update_fwd(self, pij, px, pa, ang, ang_atom, ang_i, ang_j, ln, ang_new, save_p):
        self._chk(pij, px, pa, ang, ang_atom, ang_i, ang_j, ln, ang_new, save_p)
        self._call("chg_angle_update_fwd", _p(pij), _p(px), _p(pa), _p(ang), _p(ang_atom), _p(ang_i), _p(ang_j),
                   ang_i.shape[0], _p(ln), _p(ang_new), _p(save_p))

    def angle_update_bwd(self, save_p, g_ang_in, ln, g_pre, g_ln=None):
        self._chk(save_p, g_ang_in, ln, g_pre, g_ln)
        self._call("chg_angle_update_bwd", _p(save_p), _p(g_ang_in), save_p.shape[0], _p(ln), _p(g_pre), _p(g_ln))

    # ------------------------------------------------------------------ training
    @staticmethod
    def _chk_rows(*tensors: Tensor | None) -> None:
        for t in tensors:
            if t is not None and (not t.is_cuda or t.stride(-1) != 1):
                raise ChgnetB200Error("kernel arguments must be CUDA tensors with unit column stride")

    def _workspace(self, n_out: int, device) -> Tensor:
        ws = getattr(self, "_ws", None)
        if ws is None or ws.device != device:
            need = max(int(self.lib.chg_wgrad_workspace_floats(n)) for n in (64, 128, 256))
            ws = torch.empty(need, dtype=torch.float32, device=device)
            self._ws = ws
        return ws

    def wgrad(self, x, g, out, colsum=None, x_rows=None, g_rows=None, x_silu=False, x2=None):
        self._chk_rows(x, g, out, x2)
        self._chk(colsum, x_rows, g_rows)
        if x2 is not None and x2.stride(0) != x.stride(0):
            raise ChgnetB200Error("wgrad: x2 must have the row stride of x")
        m = x_rows.shape[0] if x_rows is not None else (g_rows.shape[0] if g_rows is not None else x.shape[0])
        self._call("chg_wgrad", _p(x), _p(x2), x.stride(0), _p(x_rows), int(bool(x_silu)), _p(g), g.stride(0), _p(g_rows), m,
                   out.shape[1], _p(out), out.stride(0), _p(colsum), _p(self._workspace(out.shape[1], x.device)))

    def colsum(self, a, out, b=None, rowscale=None):
        self._chk_rows(a, b)
        self._chk(out, rowscale)
        self._call("chg_colsum", _p(a), a.stride(0), _p(b), b.stride(0) if b is not None else 0, _p(rowscale),
                   a.shape[0], a.shape[1], _p(out))

    def readout_bwd(self, x, ln, mlp_wt, mlp_w, mlp_b, w_last, seed, g_x, h_all, gz_all, g_h0, xhat):
        self._chk(x, ln, mlp_wt, mlp_w, mlp_b, w_last, seed, g_x, h_all, gz_all, g_h0, xhat)
        self._call("chg_readout_bwd", _p(x), x.shape[0], _p(ln), _p(mlp_wt), _p(mlp_w), _p(mlp_b), mlp_wt.shape[0],
                   _p(w_last), _p(seed), _p(g_x), _p(h_all), _p(gz_all), _p(g_h0), _p(xhat))

    def magmom_bwd(self, x, w, b, g_m, g_x, g_lin):
        self._chk(x, w, g_m, g_x, g_lin)
        self._call("chg_magmom_bwd", _p(x), x.shape[0], _p(w), float(b), _p(g_m), _p(g_x), _p(g_lin))

    def loss_terms(self, pred, target, kind, delta, g_pred, sums):
        self._chk(pred, target, g_pred, sums)
        self._call("chg_loss_terms", _p(pred), _p(target), pred.numel(), int(kind), float(delta), _p(g_pred), _p(sums))

    # ------------------------------------------------------------------ second order
    def edge_tangent(self, rvec, dist, rhat, center, nbr, owner, u_atom, w_graph, ddist, drhat):
        self._chk(rvec, dist, rhat, center, nbr, owner, u_atom, w_graph, ddist, drhat)
        self._call("chg_edge_tangent", _p(rvec), _p(dist), _p(rhat), _p(center), _p(nbr), _p(owner), _p(u_atom),
                   _p(w_graph), center.shape[0], _p(ddist), _p(drhat))

    def bond_basis_tangent(self, dist, ddist, u2d, freq_ag, freq_bg, rc_ag, rc_bg, p, w3t, e0d, wagd, wbgd, tbasis):
        self._chk(dist, ddist, u2d, freq_ag, freq_bg, w3t, e0d, wagd, wbgd, tbasis)
        self._call("chg_bond_basis_tangent", _p(dist), _p(ddist), _p(u2d), u2d.shape[0], _p(freq_ag), _p(freq_bg),
                   freq_ag.shape[0], float(rc_ag), float(rc_bg), int(p), _p(w3t), _p(e0d), _p(wagd), _p(wbgd), _p(tbasis))

    def bond_basis_bwd2(self, dist, ddist, u2d, freq_ag, freq_bg, rc_ag, rc_bg, p, w3, lam_e0, lam_wag, lam_wbg, g_freq):
        self._chk(dist, ddist, u2d, freq_ag, freq_bg, w3, lam_e0, lam_wag, lam_wbg, g_freq)
        self._call("chg_bond_basis_bwd2", _p(dist), _p(ddist), _p(u2d), u2d.shape[0], _p(freq_ag), _p(freq_bg),
                   freq_ag.shape[0], float(rc_ag), float(rc_bg), int(p), _p(w3), _p(lam_e0), _p(lam_wag), _p(lam_wbg),
                   _p(g_freq))

    def angle_basis_tangent(self, rhat, drhat, ang_di, ang_dj, freq, wt, a0d, tbasis):
        self._chk(rhat, drhat, ang_di, ang_dj, freq, wt, a0d, tbasis)
        self._call("chg_angle_basis_tangent", _p(rhat), _p(drhat), _p(ang_di), _p(ang_dj), ang_di.shape[0], _p(freq),
                   freq.shape[0], _p(wt), _p(a0d), _p(tbasis))

    def angle_basis_bwd2(self, rhat, drhat, ang_di, ang_dj, freq, w, lam_a0, g_freq):
        self._chk(rhat, drhat, ang_di, ang_dj, freq, w, lam_a0, g_freq)
        self._call("chg_angle_basis_bwd2", _p(rhat), _p(drhat), _p(ang_di), _p(ang_dj), ang_di.shape[0], _p(freq),
                   freq.shape[0], _p(w), _p(lam_a0), _p(g_freq))

    def atom_conv_tan(self, pcn_d, pe_d, wag, wag_d, center, nbr, d2u, save_pre, save_p, w2t, ln, msg_d, pre_d, p_d):
        self._chk(pcn_d, pe_d, wag, wag_d, center, nbr, d2u, save_pre, save_p, w2t, ln, msg_d, pre_d, p_d)
        self._call("chg_atom_conv_tan", _p(pcn_d), _p(pe_d), _p(wag), _p(wag_d), _p(center), _p(nbr), _p(d2u),
                   center.shape[0], _p(save_pre), _p(save_p), _p(w2t), _p(ln), _p(msg_d), _p(pre_d), _p(p_d))

    def atom_conv_bwd2(self, save_pre, save_p, pre_d, p_d, g_p_lam, wag, wag_d, center, d2u, lam_agg, bar_agg, w2, ln,
                       bar_pre, bar_w, u_out, g_ln):
        self._chk(save_pre, save_p, pre_d, p_d, g_p_lam, wag, wag_d, center, d2u, lam_agg, bar_agg, w2, ln, bar_pre,
                  bar_w, u_out, g_ln)
        self._call("chg_atom_conv_bwd2", _p(save_pre), _p(save_p), _p(pre_d), _p(p_d), _p(g_p_lam), _p(wag), _p(wag_d),
                   _p(center), _p(d2u), center.shape[0], _p(lam_agg), _p(bar_agg), _p(w2), _p(ln), _p(bar_pre), _p(bar_w),
                   _p(u_out), _p(g_ln))

    def bond_conv_tan(self, pij_d, px_d, pa_d, wbg, wbg_d, ang_atom, ang_i, ang_j, save_pre, save_p, w2t, ln, upd_d,
                      pre_d, p_d):
        self._chk(pij_d, px_d, pa_d, wbg, wbg_d, ang_atom, ang_i, ang_j, save_pre, save_p, w2t, ln, upd_d, pre_d, p_d)
        self._call("chg_bond_conv_tan", _p(pij_d), _p(px_d), _p(pa_d), _p(wbg), _p(wbg_d), _p(ang_atom), _p(ang_i),
                   _p(ang_j), ang_i.shape[0], _p(save_pre), _p(save_p), _p(w2t), _p(ln), _p(upd_d), _p(pre_d), _p(p_d))

    def bond_conv_bwd2(self, save_pre, save_p, pre_d, p_d, g_p_lam, wbg, wbg_d, ang_i, ang_j, lam_agg, bar_agg, w2, ln,
                       bar_pre, bar_wi, bar_wj, u_out, g_ln):
        self._chk(save_pre, save_p, pre_d, p_d, g_p_lam, wbg, wbg_d, ang_i, ang_j, lam_agg, bar_agg, w2, ln, bar_pre,
                  bar_wi, bar_wj, u_out, g_ln)
        self._call("chg_bond_conv_bwd2", _p(save_pre), _p(save_p), _p(pre_d), _p(p_d), _p(g_p_lam), _p(wbg), _p(wbg_d),
                   _p(ang_i), _p(ang_j), ang_i.shape[0], _p(lam_agg), _p(bar_agg), _p(w2), _p(ln), _p(bar_pre),
                   _p(bar_wi), _p(bar_wj), _p(u_out), _p(g_ln))

    def angle_update_tan(self, pij_d, px_d, pa_d, ang_d, ang_atom, ang_i, ang_j, save_p, ln, ang_new_d, p_d):
        self._chk(pij_d, px_d, pa_d, ang_d, ang_atom, ang_i, ang_j, save_p, ln, ang_new_d, p_d)
        self._call("chg_angle_update_tan", _p(pij_d), _p(px_d), _p(pa_d), _p(ang_d), _p(ang_atom), _p(ang_i), _p(ang_j),
                   ang_i.shape[0], _p(save_p), _p(ln), _p(ang_new_d), _p(p_d))

    def angle_update_bwd2(self, save_p, p_d, lam_ang, bar_ang, ln, bar_pre, g_ln):
        self._chk(save_p, p_d, lam_ang, bar_ang, ln, bar_pre, g_ln)
        self._call("chg_angle_update_bwd2", _p(save_p), _p(p_d), _p(lam_ang), _p(bar_ang), save_p.shape[0], _p(ln),
                   _p(bar_pre), _p(g_ln))

    def readout_bwd2(self, x, xd, ln, mlp_wt, mlp_w, mlp_b, w_last, seed, bar_x, h_all, hd_all, gz_all, zbar_all,
                     g_h0, hbar0, xhat, xhatd):
        self._chk(x, xd, ln, mlp_wt, mlp_w, mlp_b, w_last, seed, bar_x, h_all, hd_all, gz_all, zbar_all, g_h0, hbar0,
                  xhat, xhatd)
        self._call("chg_readout_bwd2", _p(x), _p(xd), x.shape[0], _p(ln), _p(mlp_wt), _p(mlp_w), _p(mlp_b),
                   mlp_wt.shape[0], _p(w_last), _p(seed), _p(bar_x), _p(h_all), _p(hd_all), _p(gz_all), _p(zbar_all),
                   _p(g_h0), _p(hbar0), _p(xhat), _p(xhatd))

    def adam_step(self, p, g, m, v, lr, beta1, beta2, eps, weight_decay, step):
        self._chk(p, g, m, v)
        self._call("chg_adam_step", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
                   float(eps), float(weight_decay), int(step))

    def readout(self, x, z, owner, ln, mlp_wt, mlp_w, mlp_b, w_last, b_last, atom_ref, site_e, h_out, e_graph,
                e_ref, g_x):
        self._chk(x, z, owner, ln, mlp_wt, mlp_w, mlp_b, w_last, atom_ref, site_e, h_out, e_graph, e_ref, g_x)
        self._call("chg_readout", _p(x), _p(z), _p(owner), x.shape[0], _p(ln), _p(mlp_wt), _p(mlp_w), _p(mlp_b),
                   mlp_wt.shape[0], _p(w_last), float(b_last), _p(atom_ref), _p(site_e), _p(h_out), _p(e_graph),
                   _p(e_ref), _p(g_x))

    def magmom(self, x, w, b, m):
        self._chk(x, w, m)
        self._call("chg_magmom", _p(x), x.shape[0], _p(w), float(b), _p(m))

    def force_virial(self, rvec, dist, rhat, g_rhat, g_dist, d2u, u2d, center, nbr, owner, force, virial):
        self._chk(rvec, dist, rhat, g_rhat, g_dist, d2u, u2d, center, nbr, owner, force, virial)
        self._call("chg_force_virial", _p(rvec), _p(dist), _p(rhat), _p(g_rhat), _p(g_dist), _p(d2u), _p(u2d),
                   _p(center), _p(nbr), _p(owner), center.shape[0], _p(force), _p(virial))
