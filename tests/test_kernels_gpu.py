"""-m gpu: every C-ABI kernel, called through ctypes with the exact arguments of a real
forward + reverse pass, against its torch specification (oracle/kernel_specs.py)."""
import numpy as np
import pytest
import torch

from chgnet_b200 import graphgen
from chgnet_b200.batch import build_batch
from chgnet_b200.engine import Engine
from chgnet_b200.weights import pack_weights

pytestmark = pytest.mark.gpu


def _record(weights, graphs, **kw):
    from kernel_replay import RecordingKernels

    sd = {k: torch.as_tensor(v) for k, v in weights.items()}
    pw = pack_weights(sd, None, device="cpu")
    rec = RecordingKernels()
    Engine(pw, rec).run(build_batch(graphs, "cpu"), **kw)
    return rec.calls


def _close(name, idx, got, want):
    got, want = got.double().cpu(), want.double()
    scale = float(want.abs().max()) if want.numel() else 1.0
    err = float((got - want).abs().max()) if want.numel() else 0.0
    # fp32 kernels vs fp32 spec: different summation order only
    tol = 2e-5 * max(scale, 1.0) + 1e-6
    assert err <= tol, f"{name} out[{idx}]: max err {err:.3e} > {tol:.3e} (scale {scale:.3e})"
    return err


@pytest.fixture(scope="module")
def recorded(weights030):
    graphs = graphgen.random_graphs(3, 10, 16, 9300)
    return _record(weights030, graphs, need_grad=True, need_magmom=True, need_atom_fea=True, need_crystal_fea=True)


@pytest.mark.parametrize("ws_min_rows", [0, 4096], ids=["tcgen05-ws-forced", "defaults-ffma"])
def test_every_kernel_matches_its_spec(recorded, ws_min_rows):
    """Both implementations of the AtomConv / BondConv entry points (warp-specialised tcgen05 3xTF32 and FFMA), and
    every other kernel, against the spec."""
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    K.set_option("ws_min_rows", ws_min_rows)  # the recorded graphs are small: 0 runs the tcgen05 kernels on them anyway
    try:
        seen = {}
        for name, snap, outs in recorded:
            args = [a.cuda() if isinstance(a, torch.Tensor) else a for a in snap]
            getattr(K, name)(*args)
            torch.cuda.synchronize()
            for idx, want in outs.items():
                err = _close(name, idx, args[idx], want)
                seen[name] = max(seen.get(name, 0.0), err)
        assert set(seen) == __import__("kernel_replay").INFER_KERNELS, sorted(seen)
        print({k: f"{v:.2e}" for k, v in seen.items()})
    finally:
        K.set_option("ws_min_rows", 4096)


def test_every_training_kernel_matches_its_spec(weights030):
    """Training reverse pass (parameter gradients): every call of a real train step, replayed."""
    import kernel_replay
    from chgnet_b200._lib import CudaKernels
    from kernel_replay import RecordingKernels

    graphs = graphgen.random_graphs(3, 10, 16, 9500)
    sd = {k: torch.as_tensor(v) for k, v in weights030.items()}
    pw = pack_weights(sd, None, device="cpu")
    rec = RecordingKernels()
    eng = Engine(pw, rec)
    out = eng.run(build_batch(graphs, "cpu"), need_grad=True, need_magmom=True, train=True)
    gen = torch.Generator().manual_seed(11)
    n_atoms = sum(g.atomic_number.shape[0] for g in graphs)
    eng.param_grads(out, torch.randn(len(graphs), generator=gen), torch.randn(n_atoms, generator=gen))
    # and a step with force / stress seeds: the second-order kernels
    out = eng.run(build_batch(graphs, "cpu"), need_grad=True, need_magmom=True, train=True)
    eng.input_grads(out, record=True)
    eng.param_grads(out, torch.randn(len(graphs), generator=gen), torch.randn(n_atoms, generator=gen),
                    torch.randn(n_atoms, 3, generator=gen), torch.randn(len(graphs), 3, 3, generator=gen))
    K = CudaKernels()
    seen = {}
    for name, snap, outs in rec.calls:
        args = [a.cuda() if isinstance(a, torch.Tensor) else a for a in snap]
        getattr(K, name)(*args)
        torch.cuda.synchronize()
        for idx, want in outs.items():
            seen[name] = max(seen.get(name, 0.0), _close(name, idx, args[idx], want))
    assert kernel_replay.TRAIN_KERNELS <= set(seen), sorted(seen)
    print({k: f"{v:.2e}" for k, v in seen.items()})


def test_loss_terms_and_adam_match_torch():
    """chg_loss_terms vs torch.nn.{MSE,L1,Huber}Loss with NaN masks (trainer.py:797-867) and
    chg_adam_step vs torch.optim.Adam (trainer.py:178-189)."""
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    g = torch.Generator(device="cuda").manual_seed(2)
    pred = torch.randn(5000, device="cuda", generator=g)
    target = pred + 0.3 * torch.randn(5000, device="cuda", generator=g)
    target[::7] = float("nan")
    valid = ~torch.isnan(target)
    for kind, crit in ((0, torch.nn.MSELoss()), (1, torch.nn.L1Loss()), (2, torch.nn.HuberLoss(delta=0.1))):
        p = pred.clone().requires_grad_(True)
        loss = crit(target[valid], p[valid])
        loss.backward()
        g_pred, sums = torch.empty_like(pred), torch.zeros(3, dtype=torch.float64, device="cuda")
        K.loss_terms(pred, target, kind, 0.1, g_pred, sums)
        n = float(sums[2])
        assert n == float(valid.sum())
        assert float(sums[0]) / n == pytest.approx(float(loss), rel=1e-5)
        assert float(sums[1]) / n == pytest.approx(float((pred - target)[valid].abs().mean()), rel=1e-5)
        assert float((g_pred / n - p.grad).abs().max()) < 1e-7
    p0 = torch.randn(100_003, device="cuda", generator=g)
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-2, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-3)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for step in range(1, 4):
        grad = torch.randn(p0.shape, device="cuda", generator=g)
        ref.grad = grad.clone()
        opt.step()
        K.adam_step(p, grad, m, v, 1e-2, 0.9, 0.999, 1e-8, 1e-3, step)
        assert float((p - ref.detach()).abs().max()) < 2e-6


@pytest.mark.parametrize("m", [1, 63, 4095, 4096, 5001, 70001], ids=lambda m: f"m={m}")
def test_linear_ragged_calls(m):
    """chg_linear on both sides of the 4096-row switch from the FFMA kernels (NT = 64 and 128) to the tensor-core
    kernels: ragged last tile, every (k, n) the model uses, bias / residual / in-place residual, and a gathered call
    (x_rows, as the engine makes for the bond-graph rows), against fp64."""
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    g = torch.Generator(device="cuda").manual_seed(5)
    for k, n in ((64, 128), (64, 256), (128, 64), (64, 64), (64, 192), (128, 128), (256, 64)):
        for has_bias, res_mode in ((True, "none"), (False, "separate"), (True, "inplace")):
            x = torch.randn(m, k, device="cuda", generator=g)
            wt = torch.randn(k, n, device="cuda", generator=g) / k ** 0.5
            bias = torch.randn(n, device="cuda", generator=g) if has_bias else None
            res = torch.randn(m, n, device="cuda", generator=g) if res_mode != "none" else None
            want = x.double() @ wt.double()
            if bias is not None:
                want += bias.double()
            if res is not None:
                want += res.double()
            y = res if res_mode == "inplace" else torch.full((m, n), float("nan"), device="cuda")
            K.linear(x, wt, bias, res, y, None, None)
            torch.cuda.synchronize()
            err = float((y.double() - want).abs().max())
            assert err < 5e-5, (m, k, n, has_bias, res_mode, err)
    x = torch.randn(2 * m + 7, 64, device="cuda", generator=g)
    rows = torch.randint(0, x.shape[0], (m,), device="cuda", generator=g, dtype=torch.int32)
    wt = torch.randn(64, 256, device="cuda", generator=g) / 8
    bias = torch.randn(256, device="cuda", generator=g)
    y = torch.full((m, 256), float("nan"), device="cuda")
    K.linear(x, wt, bias, None, y, rows)
    torch.cuda.synchronize()
    err = float((y.double() - (x.double()[rows.long()] @ wt.double() + bias.double())).abs().max())
    assert err < 5e-5, (m, "x_rows", err)


def test_kernels_without_layernorm_and_small_basis(weights030):
    """v0.2.0-shaped path: no LayerNorm, 9 radial / 9 angular functions, mlp_out bias."""
    from chgnet_b200._lib import CudaKernels
    from oracle import chgnet_oracle as orc

    args = dict(num_radial=9, num_angular=9, gMLP_norm=None, readout_norm=None, mlp_out_bias=True, cutoff_coeff=5)
    w = orc.random_weights(3, args)
    w = {k: v for k, v in w.items() if k != "mlp.layers.4.weight" and k != "mlp.layers.4.bias"}
    w["mlp.layers.5.weight"], w["mlp.layers.5.bias"] = w.pop("mlp.layers.7.weight"), w.pop("mlp.layers.7.bias")
    graphs = graphgen.random_graphs(2, 8, 12, 9400, atom_graph_cutoff=5.0)
    sd = {k: torch.as_tensor(v) for k, v in w.items()}
    from kernel_replay import RecordingKernels

    pw = pack_weights(sd, dict(atom_graph_cutoff=5.0, cutoff_coeff=5), device="cpu")
    assert not pw.hp.use_ln and pw.hp.n_readout_hidden == 2 and pw.hp.num_radial == 9
    rec = RecordingKernels()
    Engine(pw, rec).run(build_batch(graphs, "cpu", compact_bonds=False), need_grad=True, need_magmom=True)
    K = CudaKernels()
    for name, snap, outs in rec.calls:
        cargs = [a.cuda() if isinstance(a, torch.Tensor) else a for a in snap]
        getattr(K, name)(*cargs)
        for idx, want in outs.items():
            _close(name, idx, cargs[idx], want)


def test_segment_sum_strided_output_and_determinism():
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    g = torch.Generator().manual_seed(0)
    n_rows, n_items = 1000, 50000
    owners = torch.sort(torch.randint(0, n_rows, (n_items,), generator=g)).values
    ptr = torch.searchsorted(owners, torch.arange(n_rows + 1)).int().cuda()
    perm = torch.randperm(n_items, generator=g).int().cuda()
    for width in (64, 128):
        data = torch.randn(n_items, width, generator=g).cuda()
        out = torch.zeros(n_rows, 256, device="cuda")
        K.segment_sum(data, perm, ptr, 0, out[:, 64 : 64 + width])
        want = torch.zeros(n_rows, width, dtype=torch.float64).index_add_(0, owners, data[perm.long()].double().cpu())
        assert torch.allclose(out[:, 64 : 64 + width].double().cpu(), want, atol=1e-4)
        assert float(out[:, :64].abs().max()) == 0.0 and float(out[:, 64 + width :].abs().max()) == 0.0
        again = torch.zeros(n_rows, 256, device="cuda")
        K.segment_sum(data, perm, ptr, 0, again[:, 64 : 64 + width])
        assert torch.equal(out, again)  # bitwise reproducible
        K.segment_sum(data, perm, ptr, 1, again[:, 64 : 64 + width])
        assert torch.allclose(again[:, 64 : 64 + width], 2 * out[:, 64 : 64 + width], rtol=1e-6)


def test_bad_arguments_are_reported():
    from chgnet_b200._lib import ChgnetB200Error, CudaKernels

    K = CudaKernels()
    x = torch.zeros(4, 96, device="cuda")
    with pytest.raises(ChgnetB200Error, match="k must be"):
        K.linear(x, torch.zeros(96, 64, device="cuda"), None, None, torch.zeros(4, 64, device="cuda"))
    with pytest.raises(ChgnetB200Error):
        K.linear(torch.zeros(4, 64), torch.zeros(64, 64), None, None, torch.zeros(4, 64))  # CPU tensors


@pytest.mark.parametrize("m", [20011, 4095], ids=lambda m: f"m={m}")
def test_wgrad_large_reduction_matches_fp64(m):
    """chg_wgrad on both sides of the 4096-row switch from the FFMA kernel to the tensor-core kernel (csrc/wgrad_tc.cu,
    3xTF32): plain, SiLU'd and tangent activations, row gathers on either operand, strided operands, column sums -
    against fp64."""
    from chgnet_b200._lib import CudaKernels

    K = CudaKernels()
    gen = torch.Generator(device="cuda").manual_seed(5)
    # neither size is a multiple of the 64-row stage
    xs = torch.randn(m, 128, device="cuda", generator=gen)
    x2 = torch.randn(m, 128, device="cuda", generator=gen)
    gs = torch.randn(m, 256, device="cuda", generator=gen)
    perm = torch.randperm(m, device="cuda", generator=gen).int()
    sub = perm[: 9000 * m // 20011].contiguous()
    silu, dsilu = torch.nn.functional.silu, (lambda t: torch.sigmoid(t) * (1 + t * (1 - torch.sigmoid(t))))
    cases = [
        dict(x=xs[:, :64], g=gs[:, :128], n=128),
        dict(x=xs[:, 64:], g=gs[:, 64:128], n=64, x_silu=True, colsum=True),
        dict(x=xs[:, :64], g=gs[:, 128:], n=128, x2=x2[:, :64]),
        dict(x=xs[:, :64], g=gs[:, :128], n=128, x_rows=sub, colsum=True),
        dict(x=xs[:, 64:], g=gs[:, :64], n=64, g_rows=sub),
    ]
    for c in cases:
        n = c["n"]
        out = torch.empty(64, n, device="cuda")
        cs = torch.empty(n, device="cuda") if c.get("colsum") else None
        K.wgrad(c["x"], c["g"], out, cs, c.get("x_rows"), c.get("g_rows"), c.get("x_silu", False), c.get("x2"))
        torch.cuda.synchronize()
        xr = c["x"].double() if c.get("x_rows") is None else c["x"].double()[c["x_rows"].long()]
        gr = c["g"].double() if c.get("g_rows") is None else c["g"].double()[c["g_rows"].long()]
        if c.get("g_rows") is not None and c.get("x_rows") is None:
            xr = xr[: gr.shape[0]]
        if c.get("x_rows") is not None and c.get("g_rows") is None:
            gr = gr[: xr.shape[0]]
        act = xr
        if c.get("x_silu"):
            act = silu(xr)
        if c.get("x2") is not None:
            act = dsilu(xr) * c["x2"].double()
        want = act.T @ gr
        scale = float(want.abs().max())
        err = float((out.double() - want).abs().max())
        assert err < 3e-5 * scale + 1e-5, (m, c.keys(), err, scale)
        if cs is not None:
            wc = gr.sum(dim=0)
            assert float((cs.double() - wc).abs().max()) < 3e-5 * float(wc.abs().max()) + 1e-4
