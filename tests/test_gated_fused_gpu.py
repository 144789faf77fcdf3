"""The warp-specialised tcgen05 AtomConv / BondConv kernels (csrc/gated_ws.cu) and chg_segment_sum (csrc/segsum.cu)
against fp64, at the shapes where they can go wrong.

The fused forward (gated_ws_fwd_kernel + seg_stitch_kernel) reduces 16-row strips inside the CTA, writes the partials
of segments that cross a strip boundary to a workspace and adds them in a second kernel; whether that is right depends
on how segment boundaries fall against strips (16 rows), tiles (128 rows) and CTAs (one persistent CTA per SM, so
T = 128 * SMs rows is one tile per CTA).  The tests here build the segment layouts and row counts directly from seeded
generators, call the kernels through ``CudaKernels`` and compare with ``oracle.kernel_specs.SpecKernels`` run in fp64
on the same fp32 inputs.  Every output is NaN-filled before the call and followed by guard rows holding a sentinel, the
fused workspace is NaN-filled too, and every call is repeated and must give the same bits.

One test needs no GPU: it shows that the tolerance used for the aggregated messages rejects one dropped row and one
doubled strip partial, for every layout.
"""
import math

import numpy as np
import pytest
import torch

from oracle.kernel_specs import SpecKernels, _gate_fwd

B200_SMS = 148
TR, STRIP = 128, 16  # rows per tile / per reduction strip of gated_ws_fwd_kernel
WS_MIN_ROWS = 4096  # the library's default switch from the FFMA kernels to the tcgen05 kernels
GUARD = 3  # guard rows after every output
SENTINEL = -12345.0
OFFSET = 24.0  # common b2 offset of the "offset" case: LayerNorm rows with |mean| ~ 30 std

LAYOUTS = ("short", "aligned", "off_by_one", "giant", "empty_ends", "heavy_tail")

# Tolerances, as the smallest c with |got - want| <= c * scale (see _worst):
# * The second-layer GEMM is 3xTF32: a*b ~ a_hi*b_hi + a_lo*b_hi + a_hi*b_lo with a_hi = a truncated to 11 bits and
#   a_lo truncated again by the tensor core, so each product is off by at most ~3 * 2^-22 (7e-7) of |a*b|; the 64-term
#   fp32 accumulation adds at most 64 * 2^-24 (4e-6) of sum_k |h_k w_k| (DESIGN.md §4 measures 8e-6 on O(3) values).
#   C_P bounds save_p against that sum plus |b2| and |p|.
# * A message row is msg_r = o(y_r) * w_r (w: the bond weight, or the product of two for BondConv) with |do/dy| <= 1.1
#   and y = p, or LayerNorm(p) whose rows have unit scale; SiLU and sigmoid add ~2 ulp (ex2 / rcp), and the strip and
#   stitch sums at most n * 2^-24 of sum_r |msg_r| for an n-row segment.  The aggregate of segment s, column j is
#   therefore held to C_AGG * sum_r |w_rj| (|o_rj| + mean_k |o_rk|): that is sum_r |msg_rj| plus a floor that keeps
#   the column's own weight, for entries whose o happens to be near 0 while its error is not.  The bound is per
#   segment, so one wrong row of a short segment cannot hide behind a long one.  C_AGG = 2e-5 is several times the
#   per-row error above and small enough that one missing row or one doubled strip partial fails, even in a segment of
#   57k rows (test_agg_tolerance_rejects_a_dropped_row_and_a_doubled_partial).  Where LayerNorm rows have
#   |mean| >> std, p rounded to fp32 at its own magnitude moves y by ~u |mean| / std, so _c_agg adds 8 such roundings.
# * The reverse kernels are held per row: C_BWD of the row's largest |value| (same GEMM, elementwise gate algebra).
C_P = 1e-5
C_PRE = 1e-6  # save_pre: a sum of four fp32 rows, 3 roundings
C_AGG = 2e-5
C_BWD = 2e-5


def _sms() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _row_counts(sms: int) -> list[int]:
    """0 (segments but no rows), ragged single tiles, both sides of the 4096-row switch, and T, T + 1, 2T + 1, 3T + 77
    with T = 128 * SMs: the CTA that owns tile 0 runs 1, 2, 3 and 4 tiles, so both D stages are reused and every mbarrier
    parity flips."""
    t = TR * sms
    return [0, 1, 15, 16, 17, 127, 128, 129, 4095, 4096, t, t + 1, 2 * t + 1, 3 * t + 77]


ROWS = _row_counts(B200_SMS)  # the ids; the tests rebuild them from the SM count of the device they run on
ROW_IDS = ["0", "1", "15", "16", "17", "127", "128", "129", "4095", "4096", "T", "T+1", "2T+1", "3T+77"]


# ---------------------------------------------------------------------------------------------------- segment layouts
def _segment_lengths(layout: str, n_rows: int, seed: int) -> np.ndarray:
    """Lengths of consecutive segments covering exactly n_rows rows (n_rows == 0: five empty segments)."""
    rng = np.random.default_rng(seed)
    if n_rows == 0:
        return np.zeros(5, np.int64)
    if layout == "giant":  # one segment over every row, empty segments before and after it
        return np.array([0, 0, n_rows, 0, 0], np.int64)
    k = 2 * n_rows + 16
    if layout == "short":  # 0-3 rows, many per strip, 40 % empty (the BondConv shape)
        lens = rng.choice(4, size=k, p=[0.4, 0.2, 0.2, 0.2])
    elif layout == "aligned":  # 16, 32 and 128: every segment starts on a strip, every 128 on a tile
        lens = np.resize(np.array([16, 16, 32, 32, 32, 128]), k)
    elif layout == "off_by_one":  # one row short of / past a strip and a tile
        lens = np.resize(np.array([15, 17, 127, 129]), k)
    elif layout == "empty_ends":  # ptr[0] == ptr[1] ... and ptr flat at n_rows for the last segments
        lens = rng.integers(1, 48, size=k)
    elif layout == "heavy_tail":  # mostly short, some up to 300 rows
        lens = np.minimum(300, (rng.pareto(1.2, size=k) * 8).astype(np.int64))
    else:
        raise ValueError(layout)
    cs = np.cumsum(lens)
    last = int(np.searchsorted(cs, n_rows))
    lens = lens[: last + 1].astype(np.int64)
    lens[-1] -= int(cs[last]) - n_rows
    if layout == "empty_ends":
        lens = np.concatenate([np.zeros(3, np.int64), lens, np.zeros(3, np.int64)])
    assert lens.sum() == n_rows and (lens >= 0).all()
    return lens


def _ptr(lens: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).int()


def _seg_of_rows(ptr: torch.Tensor) -> torch.Tensor:
    counts = (ptr[1:] - ptr[:-1]).long()
    return torch.repeat_interleave(torch.arange(len(counts)), counts).int()


# ---------------------------------------------------------------------------------------------------- inputs
def _gated_weights(gen, variant: str, ln_on: bool):
    w2t = torch.randn(64, 128, generator=gen) / 8
    b2 = torch.randn(128, generator=gen) * 0.5
    if variant == "offset":  # |mean| ~ 30 std in every p row: the shifted one-pass LayerNorm variance
        b2 += OFFSET
    if variant == "constant":  # w2t = 0, b2 constant per half: every row of p is constant, its variance is 0
        w2t.zero_()
        b2 = torch.cat([torch.full((64,), 0.25), torch.full((64,), -0.75)])
    ln = None
    if ln_on:
        ln = torch.stack([1 + 0.1 * torch.randn(64, generator=gen), 0.1 * torch.randn(64, generator=gen),
                          1 + 0.1 * torch.randn(64, generator=gen), 0.1 * torch.randn(64, generator=gen)]).contiguous()
    return w2t, b2, ln


def _saturated_rows(n_rows: int) -> torch.Tensor:
    """A few rows, spread over the call and including the first and last, whose pre-activations are about +-60."""
    return torch.unique(torch.linspace(0, max(n_rows - 1, 0), 9).round().long())


def _inputs(mode: str, ptr: torch.Tensor, variant: str, ln_on: bool, seed: int) -> dict:
    """CPU fp32 / int32 arguments of chg_atom_conv_fused ("atom") or chg_bond_conv_fused ("bond")."""
    gen = torch.Generator().manual_seed(seed)
    seg = _seg_of_rows(ptr)
    n_rows, n_seg = seg.shape[0], ptr.shape[0] - 1
    w2t, b2, ln = _gated_weights(gen, variant, ln_on)
    sat = _saturated_rows(n_rows) if variant == "saturated" and n_rows else None
    if mode == "atom":
        n_atoms, n_und = n_seg, max(1, n_rows // 2 + 7)  # segment = centre atom
        a = dict(pcn=torch.randn(n_atoms, 256, generator=gen) * 0.5, pe=torch.randn(n_und, 128, generator=gen) * 0.5,
                 wag=torch.randn(n_und, 64, generator=gen), center=seg,
                 nbr=torch.randint(0, n_atoms, (n_rows,), generator=gen).int(),
                 d2u=torch.randint(0, n_und, (n_rows,), generator=gen).int())
        if sat is not None:  # these rows read extra pe rows of +-60 (the first half all -60: SiLU of the gather ~ 0)
            big = 60.0 * torch.sign(torch.randn(len(sat), 128, generator=gen))
            big[: len(sat) // 2] = -60.0
            a["pe"] = torch.cat([a["pe"], big])
            a["d2u"][sat] = (n_und + torch.arange(len(sat))).int()
            a["wag"] = torch.cat([a["wag"], torch.randn(len(sat), 64, generator=gen)])
    else:
        n_slots, n_atoms = n_seg, max(1, n_rows // 8 + 3)  # segment = bond slot i
        a = dict(pij=torch.randn(n_slots, 256, generator=gen) * 0.4, px=torch.randn(n_atoms, 128, generator=gen) * 0.4,
                 pa=torch.randn(n_rows, 128, generator=gen) * 0.4, wbg=torch.randn(n_slots, 64, generator=gen),
                 ang_atom=torch.randint(0, n_atoms, (n_rows,), generator=gen).int(), ang_i=seg,
                 ang_j=torch.randint(0, n_slots, (n_rows,), generator=gen).int())
        if sat is not None:
            big = 60.0 * torch.sign(torch.randn(len(sat), 128, generator=gen))
            big[: len(sat) // 2] = -60.0
            a["pa"][sat] = big
    a.update(ptr=ptr, w2t=w2t, b2=b2, ln=ln)
    return a


def _d(t):
    return None if t is None else (t.double() if t.is_floating_point() else t)


def _spec_forward(mode: str, a: dict) -> dict:
    """fp64 spec of the message per row, its aggregate, |message| aggregated, p, pre and the scales of p and pre."""
    S = SpecKernels()
    d = {k: _d(v) for k, v in a.items()}
    n, n_seg = a["center" if mode == "atom" else "ang_i"].shape[0], a["ptr"].shape[0] - 1
    msg, p, pre = (torch.empty(n, w, dtype=torch.float64) for w in (64, 128, 128))
    if mode == "atom":
        S.atom_conv_fwd(d["pcn"], d["pe"], d["wag"], a["center"], a["nbr"], a["d2u"], d["w2t"], d["b2"], d["ln"], msg, p, pre)
        pre_scale = S._atom_pre(d["pcn"].abs(), d["pe"].abs(), a["center"], a["nbr"], a["d2u"])
    else:
        S.bond_conv_fwd(d["pij"], d["px"], d["pa"], d["wbg"], a["ang_atom"], a["ang_i"], a["ang_j"], d["w2t"], d["b2"],
                        d["ln"], msg, pre, p)
        pre_scale = S._bond_pre(d["pij"].abs(), d["px"].abs(), d["pa"].abs(), a["ang_atom"], a["ang_i"], a["ang_j"])
    h, w = torch.nn.functional.silu(pre).abs(), d["w2t"].abs()
    p_scale = torch.cat([h[:, :64] @ w[:, :64], h[:, 64:] @ w[:, 64:]], dim=1) + d["b2"].abs() + p.abs()
    # msg = o * weight: the per-row magnitude |weight| * (|o| + the row's mean |o|) is |msg| plus a floor that keeps
    # the column's own weight, for entries whose o happens to be near 0 while its error is not
    o = _gate_fwd(p, d["ln"])[0].abs()
    if mode == "atom":
        wrow = d["wag"][a["d2u"].long()]
    else:
        wrow = d["wbg"][a["ang_i"].long()] * d["wbg"][a["ang_j"].long()]
    seg = _seg_of_rows(a["ptr"]).long()
    agg = torch.zeros(n_seg, 64, dtype=torch.float64).index_add_(0, seg, msg)
    mag = torch.zeros(n_seg, 64, dtype=torch.float64).index_add_(0, seg, wrow.abs() * (o + o.mean(dim=1, keepdim=True)))
    # LayerNorm divides by the row's std: p rounded to fp32 at its own magnitude moves y by ~u |mean| / std
    halves = p.view(-1, 2, 64)
    mean, std = halves.mean(dim=2), halves.std(dim=2, unbiased=False)
    cond = (mean.abs() / std)[std > 0]  # rows of constant p (std 0) are exact
    ln_cond = float(cond.max()) if d["ln"] is not None and cond.numel() else 0.0
    return dict(msg=msg, agg=agg, mag=mag, p=p, pre=pre, p_scale=p_scale, pre_scale=pre_scale, ln_cond=ln_cond)


def _c_agg(want: dict) -> float:
    """C_AGG, plus 8 fp32 roundings of p relative to the LayerNorm row's std where rows have |mean| >> std."""
    return C_AGG + 8 * 2.0**-24 * want["ln_cond"]


# ---------------------------------------------------------------------------------------------------- comparisons
def _worst(got: torch.Tensor, want: torch.Tensor, scale: torch.Tensor) -> float:
    """The smallest c with |got - want| <= c * scale everywhere: inf where got is NaN or inf, or where it differs from
    want at all where scale is 0 (an empty segment must be exactly 0)."""
    if want.numel() == 0:
        return 0.0
    err = (got.detach().double().cpu() - want).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / scale.expand_as(err))
    return float(torch.nan_to_num(ratio, nan=math.inf, posinf=math.inf).max())


def _agg_worst(got: torch.Tensor, want: torch.Tensor, mag: torch.Tensor) -> float:
    """_worst of an aggregate against C_AGG's scale: mag = per segment and column, sum_r |w_r| (|o_r| + mean |o_r|)."""
    return _worst(got, want, mag)


def _row_scale(want: torch.Tensor) -> torch.Tensor:
    return want.abs().amax(dim=1, keepdim=True) if want.numel() else want


def _guarded(rows: int, cols: int, fill: float = math.nan) -> tuple[torch.Tensor, torch.Tensor]:
    """(buffer, view): `rows` rows of `fill` followed by GUARD rows of SENTINEL; the view is the first `rows` rows."""
    buf = torch.full((rows + GUARD, cols), SENTINEL, device="cuda")
    buf[:rows] = fill
    return buf, buf[:rows]


def _guards_intact(buf: torch.Tensor, rows: int, name: str) -> None:
    assert bool((buf[rows:] == SENTINEL).all()), f"{name}: a guard row after row {rows} was written"


def _gpu(a: dict) -> dict:
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in a.items()}


def _run_fused(K, mode: str, g: dict, n_rows: int, n_seg: int, with_saves: bool) -> dict:
    """One fused call on NaN-filled, guarded outputs and a NaN-filled (guarded) workspace; returns the outputs."""
    need = int(K.lib.chg_gated_fused_workspace_floats(n_rows))
    ws = torch.full((need + 64,), math.nan, device="cuda")
    ws[need:] = SENTINEL
    K._fws = ws  # CudaKernels._fused_work reuses a buffer that is large enough
    agg_buf, agg = _guarded(n_seg, 64)
    sp_buf, save_p = _guarded(n_rows, 128) if with_saves else (None, None)
    spre_buf, save_pre = _guarded(n_rows, 128) if with_saves and mode == "bond" else (None, None)
    if mode == "atom":
        K.atom_conv_fused(g["pcn"], g["pe"], g["wag"], g["center"], g["nbr"], g["d2u"], g["ptr"], g["w2t"], g["b2"], g["ln"],
                          agg, save_p)
    else:
        K.bond_conv_fused(g["pij"], g["px"], g["pa"], g["wbg"], g["ang_atom"], g["ang_i"], g["ang_j"], g["ptr"], g["w2t"],
                          g["b2"], g["ln"], agg, save_pre, save_p)
    torch.cuda.synchronize()
    assert K._fws is ws and bool((ws[need:] == SENTINEL).all()), "the fused kernels wrote past their workspace"
    _guards_intact(agg_buf, n_seg, "agg")
    out = dict(agg=agg.clone())
    if with_saves:
        _guards_intact(sp_buf, n_rows, "save_p")
        out["save_p"] = save_p.clone()
        if mode == "bond":
            _guards_intact(spre_buf, n_rows, "save_pre")
            out["save_pre"] = save_pre.clone()
    return out


def _paths(n_rows: int) -> list[tuple[str, int]]:
    """(label, ws_min_rows) of the implementations to run: the tcgen05 kernels are forced below 4096 rows; at 4095 and
    4096 both the default choice and the other implementation run, so both sides of the switch agree with fp64."""
    if n_rows == 0:
        return [("tcgen05", 0), ("ffma", WS_MIN_ROWS)]
    if n_rows in (4095, 4096):
        return [("default", WS_MIN_ROWS), ("tcgen05" if n_rows < WS_MIN_ROWS else "ffma", 0 if n_rows < WS_MIN_ROWS else n_rows + 1)]
    if n_rows < WS_MIN_ROWS:
        return [("tcgen05", 0)]
    return [("default", WS_MIN_ROWS)]


def _check_fused(mode: str, n_rows: int, layout: str, variant: str, ln_on: bool, with_saves: bool, seed: int) -> dict:
    from chgnet_b200._lib import CudaKernels

    ptr = _ptr(_segment_lengths(layout, n_rows, seed))
    n_seg = ptr.shape[0] - 1
    a = _inputs(mode, ptr, variant, ln_on, seed + 1)
    want = _spec_forward(mode, a)
    g = _gpu(a)
    K = CudaKernels()
    worst = {}
    try:
        for label, ws_min in _paths(n_rows):
            K.set_option("ws_min_rows", ws_min)
            first = _run_fused(K, mode, g, n_rows, n_seg, with_saves)
            again = _run_fused(K, mode, g, n_rows, n_seg, with_saves)
            for k in first:
                assert torch.equal(first[k], again[k]), f"{label}: {k} differs between two identical calls"
            w = {"agg": _agg_worst(first["agg"], want["agg"], want["mag"])}
            if with_saves:
                w["save_p"] = _worst(first["save_p"], want["p"], want["p_scale"])
                if mode == "bond":
                    w["save_pre"] = _worst(first["save_pre"], want["pre"], want["pre_scale"])
            if n_rows == 0:
                assert float(first["agg"].abs().max()) == 0.0, f"{label}: no rows, but a non-zero aggregate"
            worst[label] = w
    finally:
        K.set_option("ws_min_rows", WS_MIN_ROWS)
    print(f"{mode} ln={ln_on} rows={n_rows} layout={layout} variant={variant} saves={with_saves}:",
          {lab: {k: f"{v:.1e}" for k, v in w.items()} for lab, w in worst.items()})
    for label, w in worst.items():
        assert w["agg"] <= _c_agg(want), (label, "agg", w["agg"], _c_agg(want))
        assert w.get("save_p", 0.0) <= C_P, (label, "save_p", w["save_p"])
        assert w.get("save_pre", 0.0) <= C_PRE, (label, "save_pre", w["save_pre"])
    return worst


# ---------------------------------------------------------------------------------------------------- 1. fused forward
@pytest.mark.gpu
@pytest.mark.parametrize("ln_on", [True, False], ids=["ln", "no-ln"])
@pytest.mark.parametrize("mode", ["atom", "bond"])
@pytest.mark.parametrize("i", range(len(ROWS)), ids=ROW_IDS)
def test_fused_forward_matches_fp64(mode, ln_on, i):
    """chg_atom_conv_fused / chg_bond_conv_fused at every row count of _row_counts.  The layout rotates with the row
    count (shifted by 4 between the LayerNorm settings), so each mode meets all six layouts at the multi-tile counts
    T .. 3T + 77 and at least twice among the rest; the saved p / pre are requested on every other row count."""
    n_rows = _row_counts(_sms())[i]
    layout = LAYOUTS[(i + (4 if ln_on else 0)) % len(LAYOUTS)]
    _check_fused(mode, n_rows, layout, "plain", ln_on, with_saves=(i + ln_on) % 2 == 0, seed=100 * i + 7 * ln_on)


@pytest.mark.gpu
@pytest.mark.parametrize("ln_on", [True, False], ids=["ln", "no-ln"])
@pytest.mark.parametrize("mode", ["atom", "bond"])
@pytest.mark.parametrize("variant", ["offset", "constant", "saturated"])
def test_fused_forward_numerics(mode, ln_on, variant):
    """At T + 1 rows (two tiles on the first CTA), heavy-tailed segments: a b2 offset that makes |mean| >> std in every
    LayerNorm row (the epilogue's shifted one-pass variance), rows of constant p (variance 0, the fmaxf clamp), and a
    few rows with |pre| ~ 60 where the ex2 / rcp of SiLU and sigmoid saturate."""
    n_rows = TR * _sms() + 1
    _check_fused(mode, n_rows, "heavy_tail", variant, ln_on, with_saves=True, seed=5000 + len(variant))


# ---------------------------------------------------------------------------------------------------- tolerance check
@pytest.mark.parametrize("mode", ["atom", "bond"])
def test_agg_tolerance_rejects_a_dropped_row_and_a_doubled_partial(mode):
    """CPU: the comparison the fused-forward tests use (_agg_worst <= C_AGG) is tight enough to catch the failures a
    strip reduction can have.  For every layout at 3T + 77 rows (B200), take the fp64 spec aggregate, then (a) drop one
    row of a segment that spans several strips and (b) add one of its 16-row strip partials a second time: both must
    be rejected, while the exact aggregate passes."""
    n_rows = 3 * TR * B200_SMS + 77
    rng = np.random.default_rng(17)
    for li, layout in enumerate(LAYOUTS):
        ptr = _ptr(_segment_lengths(layout, n_rows, 300 + li))
        want = _spec_forward(mode, _inputs(mode, ptr, "plain", True, 301 + li))
        assert _agg_worst(want["agg"], want["agg"], want["mag"]) == 0.0
        p = ptr.long().numpy()
        multi = [s for s in range(len(p) - 1) if p[s + 1] > p[s] and p[s] // STRIP != (p[s + 1] - 1) // STRIP]
        assert multi, layout
        s = int(rng.choice(multi))
        lo, hi = int(p[s]), int(p[s + 1])
        r = int(rng.integers(lo, hi))
        dropped = want["agg"].clone()
        dropped[s] -= want["msg"][r]
        k = int(rng.integers(lo // STRIP, (hi - 1) // STRIP + 1))
        doubled = want["agg"].clone()
        doubled[s] += want["msg"][max(lo, k * STRIP) : min(hi, (k + 1) * STRIP)].sum(dim=0)
        w_drop = _agg_worst(dropped, want["agg"], want["mag"])
        w_double = _agg_worst(doubled, want["agg"], want["mag"])
        c = _c_agg(want)
        print(f"{mode} {layout}: segment of {hi - lo} rows; dropped row -> {w_drop:.1e}, doubled strip {k} -> "
              f"{w_double:.1e} (tolerance {c:.1e})")
        assert w_drop > c, (layout, hi - lo, w_drop, c)
        assert w_double > c, (layout, hi - lo, w_double, c)


# ---------------------------------------------------------------------------------------------------- 2. reverse
@pytest.mark.gpu
@pytest.mark.parametrize("ln_on", [True, False], ids=["ln", "no-ln"])
@pytest.mark.parametrize("mode", ["atom", "bond"])
@pytest.mark.parametrize("i", range(len(ROWS)), ids=ROW_IDS)
def test_ws_reverse_matches_fp64(mode, ln_on, i):
    """chg_atom_conv_bwd / chg_bond_conv_bwd in inference form (g_p = g_ln = None) at every row count of _row_counts:
    save_p / save_pre come from the fp64 spec forward cast to fp32, g_agg is random, so this does not depend on the
    forward kernels.  g_pre, g_w (AtomConv) and gw_i / gw_j (BondConv) against the fp64 spec, row by row."""
    from chgnet_b200._lib import CudaKernels

    n_rows = _row_counts(_sms())[i]
    seed = 900 + 100 * i + 7 * ln_on
    ptr = _ptr(_segment_lengths(LAYOUTS[(i + 3 * ln_on) % len(LAYOUTS)], n_rows, seed))
    n_seg = ptr.shape[0] - 1
    a = _inputs(mode, ptr, "plain", ln_on, seed + 1)
    fwd = _spec_forward(mode, a)
    gen = torch.Generator().manual_seed(seed + 2)
    a.update(save_p=fwd["p"].float(), save_pre=fwd["pre"].float(), g_agg=torch.randn(n_seg, 64, generator=gen),
             w2=a["w2t"].t().contiguous())
    d = {k: _d(v) for k, v in a.items()}
    S = SpecKernels()
    want = {"g_pre": torch.empty(n_rows, 128, dtype=torch.float64)}
    if mode == "atom":
        want["g_w"] = torch.empty(n_rows, 64, dtype=torch.float64)
        S.atom_conv_bwd(d["pcn"], d["pe"], d["wag"], a["center"], a["nbr"], a["d2u"], d["save_p"], d["g_agg"], d["w2"],
                        d["ln"], want["g_pre"], want["g_w"])
    else:
        want["gw_i"], want["gw_j"] = torch.empty(n_rows, 64, dtype=torch.float64), torch.empty(n_rows, 64, dtype=torch.float64)
        S.bond_conv_bwd(d["save_pre"], d["save_p"], d["wbg"], a["ang_i"], a["ang_j"], d["g_agg"], d["w2"], d["ln"],
                        want["g_pre"], want["gw_i"], want["gw_j"])
    g = _gpu(a)
    K = CudaKernels()
    worst = {}
    try:
        for label, ws_min in _paths(n_rows):
            K.set_option("ws_min_rows", ws_min)
            runs = []
            for _ in range(2):
                bufs = {k: _guarded(n_rows, v.shape[1]) for k, v in want.items()}
                o = {k: view for k, (_, view) in bufs.items()}
                if mode == "atom":
                    K.atom_conv_bwd(g["pcn"], g["pe"], g["wag"], g["center"], g["nbr"], g["d2u"], g["save_p"], g["g_agg"],
                                    g["w2"], g["ln"], o["g_pre"], o["g_w"])
                else:
                    K.bond_conv_bwd(g["save_pre"], g["save_p"], g["wbg"], g["ang_i"], g["ang_j"], g["g_agg"], g["w2"],
                                    g["ln"], o["g_pre"], o["gw_i"], o["gw_j"])
                torch.cuda.synchronize()
                for k, (buf, _) in bufs.items():
                    _guards_intact(buf, n_rows, k)
                runs.append({k: v.clone() for k, v in o.items()})
            for k in want:
                assert torch.equal(runs[0][k], runs[1][k]), f"{label}: {k} differs between two identical calls"
            worst[label] = {k: _worst(runs[0][k], want[k], _row_scale(want[k])) for k in want}
    finally:
        K.set_option("ws_min_rows", WS_MIN_ROWS)
    print(f"{mode} ln={ln_on} rows={n_rows}:", {lab: {k: f"{v:.1e}" for k, v in w.items()} for lab, w in worst.items()})
    for label, w in worst.items():
        for k, v in w.items():
            assert v <= C_BWD, (label, k, v)


# ---------------------------------------------------------------------------------------------------- 3. segment_sum
def _lane_groups(width: int, n_rows: int, n_items: int, sms: int) -> int:
    """The lane-groups per output row chg_segment_sum picks (csrc/segsum.cu), restated:
        avg = n_items / n_rows (integer), groups = 256 / (width / 4) lane-groups per CTA, resident = 8 * SMs CTAs;
        S = 1; while S < 8 and avg >= 16 S and ceil(n_rows * 2S / groups) <= resident: S *= 2
        if S == 1 and avg >= 32: S = 2
    One CTA pass covers groups / S output rows; the grid is min(passes, resident) CTAs, so a CTA loops over more than
    one pass only when n_rows > resident * groups / S.  S = 4 and 8 are only chosen when every pass fits one wave, so
    the multi-pass points below are S = 1 and the S = 2 that the last line picks."""
    avg, groups, resident = n_items // n_rows, 256 // (width // 4), 8 * sms
    s = 1
    while s < 8 and avg >= 16 * s and (n_rows * 2 * s + groups - 1) // groups <= resident:
        s *= 2
    if s == 1 and avg >= 32:
        s = 2
    return s


def _segsum_points(width: int, sms: int) -> list[tuple[int, int, int]]:
    """(expected S, n_rows, mean segment length).  Odd row counts leave the last pass partly past n_rows (r >= n_rows
    for some lane-groups) whenever a pass covers more than one row."""
    g, res = 256 // (width // 4), 8 * sms
    return [
        (1, 2 * g * res + 5, 8),  # mean < 16; n_rows / g > resident passes: CTAs loop
        (2, g * res // 2 - 3, 24),  # 16 <= mean < 32, n_rows * 2 / g <= resident: one wave
        (2, g * res + 3, 40),  # mean >= 32 but too many rows for one wave at S = 2: the fallback S = 2, CTAs loop
        (4, g * res // 4 - 1, 48),  # 32 <= mean < 64, n_rows * 4 / g <= resident
        (8, g * res // 8 - 1, 100),  # mean >= 64, n_rows * 8 / g <= resident
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("point", range(5), ids=["S1-multipass", "S2", "S2-multipass", "S4", "S8"])
def test_segment_sum_every_lane_group_count(width, point):
    """chg_segment_sum at a point of each lane-group count S, both widths: with and without perm, accumulate 0 and 1,
    into a strided view with guard rows and columns, with empty segments (the first, ~10 % of the rest and the last
    five) - against an fp64 index_add_, and bitwise equal on a second call."""
    from chgnet_b200._lib import CudaKernels

    sms = _sms()
    want_s, n_rows, mean = _segsum_points(width, sms)[point]
    rng = np.random.default_rng(40 + point)
    lens = rng.integers(0, 2 * mean + 1, size=n_rows)
    lens[rng.random(n_rows) < 0.1] = 0
    lens[0], lens[-5:] = 0, 0
    n_items = int(lens.sum())
    s = _lane_groups(width, n_rows, n_items, sms)
    assert s == want_s, (width, n_rows, n_items, s)
    rows_per_pass = 256 // (width // 4) // s
    passes = -(-n_rows // rows_per_pass)
    assert (passes > 8 * sms) == (point in (0, 2)), (passes, 8 * sms)
    ptr = _ptr(lens)
    owner = _seg_of_rows(ptr).long()
    seg_len = torch.from_numpy(lens).double()[:, None]
    gen = torch.Generator().manual_seed(60 + point)
    extra = 1000
    data = torch.randn(n_items + extra, width, generator=gen)
    perm = torch.randperm(n_items + extra, generator=gen)[:n_items].int()
    init = torch.randn(n_rows, width, generator=gen)
    K = CudaKernels()
    gd, gp, gptr = data.cuda(), perm.cuda(), ptr.cuda()
    u = 2.0**-24
    for use_perm in (False, True):
        src = (data[perm.long()] if use_perm else data[:n_items]).double()
        sums = torch.zeros(n_rows, width, dtype=torch.float64).index_add_(0, owner, src)
        mag = torch.zeros(n_rows, width, dtype=torch.float64).index_add_(0, owner, src.abs())
        for accumulate in (0, 1):
            want = sums + init.double() if accumulate else sums
            # recursive fp32 summation of n terms: |error| <= (n - 1) u sum |x|; one more rounding when accumulating
            scale = (seg_len + 2) * u * (mag + (init.double().abs() if accumulate else 0.0))
            outs = []
            for _ in range(2):
                buf = torch.full((n_rows + GUARD, 256), SENTINEL, device="cuda")
                view = buf[:n_rows, 64 : 64 + width]
                view.copy_(init if accumulate else torch.full_like(init, math.nan))
                K.segment_sum(gd if use_perm else gd[:n_items], gp if use_perm else None, gptr, accumulate, view)
                torch.cuda.synchronize()
                assert bool((buf[:, :64] == SENTINEL).all()) and bool((buf[:, 64 + width :] == SENTINEL).all())
                _guards_intact(buf, n_rows, "out")
                outs.append(view.clone())
            assert torch.equal(outs[0], outs[1]), (use_perm, accumulate)
            worst = _worst(outs[0], want, scale)
            print(f"width {width} S={s} rows={n_rows} items={n_items} perm={use_perm} acc={accumulate}: "
                  f"worst {worst:.2f} of the fp32 summation bound")
            assert worst <= 1.0, (use_perm, accumulate, worst)
