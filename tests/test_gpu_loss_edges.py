"""The large-tile contrastive-loss kernels off the benchmarked point, against the fp64 oracle.

From 4096 x 4096 logits on, the statistics come from rowsweep_kernel and the stored-weights gradient from
rowgrad_kernel + colgrad_kernel, with pair_kernel<kBwdP> / <kBwdW> adding the flagged tiles.  test_gpu_loss.py checks
them at B = 8192 / 32768, D = 256, tau = 1 on LayerNorm-scale rows.  This module checks them where kernels go wrong:

* ragged batches (B mod 128 in {1, 127}, B mod 256 on both sides of 128), both embedding widths, concentrated and soft
  targets (the device-side gate takes the stored-weights form for the first and the own-rows sweep for the second);
* a batch whose row statistics are far negative and span ~200 binades (images in a cone, three captions on its far
  side): the padded columns of a ragged last tile then meet fp16 weights near overflow, and the wide-range ("slow")
  exponential path runs;
* temperatures other than 1, through the fused step, the sharded stored-weights form and the column-partials statistics;
* the wide-range exponential path at the large-tile sizes (rows of very different norm);
* an upstream gradient other than 1 through the phased stored-weights and own-rows forms.

Every case asserts which path ran (the gate's choice of gradient form, the span of the statistics that selects the
exponential path) and checks, besides the whole-tensor bars of test_gpu_loss.py, every 128-row block of dI and dT on
its own: an error confined to one tile (a ragged last block, a last strip, one column split) hardly moves a whole-tensor
norm."""
import numpy as np
import pytest
import torch

from _loss_phases import _phases, _phases_sharded
from conftest import rel_err
from oracle import loss_blockwise, loss_ref

pytestmark = pytest.mark.gpu

MODES = ["tc_f16x3", "tc_f16"]
# whole-tensor bars (BASELINE.json north_star; the single-pass engine's stated looser ones): loss, gradients
TOLS = {"tc_f16x3": (1e-4, 1e-3), "tc_f16": (5e-4, 5e-3)}
# Per-128-row-block bar on dI and dT.  Largest block error measured over this module (NVIDIA B200, 1000 W power limit;
# the kernels are bit-deterministic): 7.3e-4 for tc_f16x3 (tau = 2, B = 8192, fused step) and 1.1e-3 for tc_f16 (the
# cone batch, B = 8191); the bars leave 1.6x / 1.8x of headroom.  A block that is 1 % off reads as >= 1e-2, 8x / 5x
# above them.
BLOCK_TOL = {"tc_f16x3": 1.2e-3, "tc_f16": 2e-3}
# the length-B statistics vectors (row / column LSE of S, row LSE of Z: as test_gpu_loss.py's column-partials test;
# g_i = sum_j P_ij G_ij and q_i = colsum(P)_i: the loss bars)
STAT_TOLS = {"tc_f16x3": (2e-5, 1e-4), "tc_f16": (2e-3, 5e-4)}
LOG2E = 1.4426950408889634
FAST_PATH_BINADES = 60.0    # wscale_kernel: statistics spanning more than this take the wide-range exponential path


# ------------------------------------------------------------------ batches
def _layernorm_batch(B, D, scale, seed=0):
    """LayerNorm'd gaussian rows (what ProjectionHead emits) times `scale`: 1.0 concentrated soft targets (diagonal
    tiles only), 0.25 soft ones (every tile flagged)."""
    I = loss_ref.make_embeddings(B, D, seed=1000 + seed, scale=scale)
    T = loss_ref.make_embeddings(B, D, seed=5000 + seed, scale=scale)
    return I, T


def _cone_batch(B, opposite_images=False):
    """Images in a cone around a fixed direction u (|u| = 16, zero mean): I = 0.6 u + 0.8 (LayerNorm row), and the
    captions of rows 0-2 on its far side, T_k = -(0.6 u + 0.8 T_k).  Those rows get row LSE r_k ~ -50 and the
    statistics span ~200 binades.  `opposite_images` swaps the towers: three images opposite a cone of captions, whose
    COLUMN LSE c_k is then the far negative one."""
    I = loss_ref.make_embeddings(B, 256, seed=1).double()
    T = loss_ref.make_embeddings(B, 256, seed=2).double()
    u = torch.from_numpy(np.random.default_rng(3).standard_normal(256))
    u = (u - u.mean()) * (16.0 / (u - u.mean()).norm())
    I = 0.6 * u + 0.8 * I
    T[:3] = -(0.6 * u + 0.8 * T[:3])
    I, T = I.float(), T.float()
    return (T, I) if opposite_images else (I, T)


def _wide_norm_batch(B):
    """Rows of very different norm (x 0.05 ... x 1, shuffled), as test_gpu_loss.py's test_loss_wide_norm_spread."""
    g = torch.Generator().manual_seed(5)
    w = torch.logspace(-1.3, 0.0, B)[torch.randperm(B, generator=g)].unsqueeze(1)
    I = loss_ref.make_embeddings(B, 256, seed=12, scale=1.0) * w
    T = loss_ref.make_embeddings(B, 256, seed=13, scale=1.0) * w
    return I, T


# ------------------------------------------------------------------ reference
_ORACLE = {}


def _oracle(key, I, T, tau, grad_loss=1.0):
    """fp64 loss, gradients and statistics: the blockwise oracle (plain torch fp64 on the GPU) from 4096 rows on, the
    numpy closed form below.  One batch is kept between the tests of one case."""
    key = (key, tau, grad_loss)
    if key not in _ORACLE:
        _ORACLE.clear()
        if I.shape[0] >= 4096:
            loss, dI, dT, st = loss_blockwise.clip_loss_blockwise_f64(I.cuda(), T.cuda(), tau, rows=1024, grad_loss=grad_loss)
            st = {k: v.cpu() for k, v in st.items()}
            dI, dT = dI.cpu(), dT.cpu()
        else:
            loss, dI, dT, st = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), tau, grad_loss=grad_loss)
            dI, dT = torch.from_numpy(dI), torch.from_numpy(dT)
            st = {k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}
        _ORACLE[key] = (float(loss), dI, dT, st)
    return _ORACLE[key]


def _span_binades(st):
    """The span wscale_kernel tests: row and column LSE of S together, and the row LSE of Z (the larger one)."""
    rc = torch.cat([st["row_lse_s"], st["col_lse_s"]])
    rz = st["row_lse_z"]
    return max((rc.max() - rc.min()).item(), (rz.max() - rz.min()).item()) * LOG2E


def _exp_path(st):
    """Which exponential path the gradient kernels take for these statistics: "fast" (factored) or "wide".  The span
    must be a binade away from the threshold, so that the device's fp32 statistics cannot choose the other one."""
    span = _span_binades(st)
    assert abs(span - FAST_PATH_BINADES) > 1.0, span
    return "fast" if span < FAST_PATH_BINADES else "wide"


# ------------------------------------------------------------------ metric
def _block_errors(d, ref, rows=128):
    """Relative error of every `rows`-row block: ||d_k - ref_k|| / ||ref_k||, on RMS values so that a ragged last block
    weighs like a full one.  A block whose reference RMS is below a tenth of the median block's is measured against
    that tenth (its own norm would turn rounding noise into a large ratio).  Returns (errors, floor RMS)."""
    d = torch.as_tensor(d).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    B, D = ref.shape
    nb = (B + rows - 1) // rows
    pad = nb * rows - B
    diff = torch.nn.functional.pad(d - ref, (0, 0, 0, pad)).reshape(nb, rows * D).norm(dim=1)
    rn = torch.nn.functional.pad(ref, (0, 0, 0, pad)).reshape(nb, rows * D).norm(dim=1)
    n = torch.full((nb,), float(rows), dtype=torch.float64)
    n[-1] = B - (nb - 1) * rows
    rms = rn / n.sqrt()
    floor = 0.1 * rms.median()
    return (diff / n.sqrt()) / torch.maximum(rms, floor), floor


def _rows_error(d, ref, idx, floor):
    d = torch.as_tensor(d).double().cpu()[idx]
    ref = torch.as_tensor(ref).double().cpu()[idx]
    return (d - ref).norm().item() / max(ref.norm().item(), floor.item() * len(idx) ** 0.5)


def _check(label, mode, loss, dI, dT, ref, rows=()):
    """Finite outputs; loss and whole-tensor gradient bars; every 128-row block of dI and dT (the ragged last one and
    the rows the case names reported on their own)."""
    ref_loss, ref_dI, ref_dT, _st = ref
    dI, dT = torch.as_tensor(dI).cpu(), torch.as_tensor(dT).cpu()
    assert np.isfinite(loss), (label, loss)
    bad = [name for name, g in (("dI", dI), ("dT", dT)) if not bool(torch.isfinite(g).all())]
    assert not bad, f"{label} {mode}: non-finite rows of {bad}: " + ", ".join(
        f"{name} {torch.nonzero(~torch.isfinite(g).all(dim=1)).flatten()[:8].tolist()}"
        for name, g in (("dI", dI), ("dT", dT)) if name in bad)
    lt, gt = TOLS[mode]
    el = abs(loss - ref_loss) / abs(ref_loss)
    eI, eT = rel_err(dI, ref_dI), rel_err(dT, ref_dT)
    bI, fI = _block_errors(dI, ref_dI)
    bT, fT = _block_errors(dT, ref_dT)
    row_errs = [_rows_error(dI, ref_dI, list(rows), fI), _rows_error(dT, ref_dT, list(rows), fT)] if rows else []
    print(f"edges {label} {mode}: loss {el:.1e} whole dI {eI:.2e} dT {eT:.2e} | block max dI {bI.max():.2e} "
          f"(#{int(bI.argmax())}) dT {bT.max():.2e} (#{int(bT.argmax())}) | last dI {bI[-1]:.2e} dT {bT[-1]:.2e}"
          + (f" | rows {list(rows)} dI {row_errs[0]:.2e} dT {row_errs[1]:.2e}" if rows else ""))
    assert el <= lt, (label, mode, loss, ref_loss)
    assert eI < gt and eT < gt, (label, mode, eI, eT)
    bt = BLOCK_TOL[mode]
    assert bI.max() < bt and bT.max() < bt, (label, mode, "block", int(bI.argmax()), bI.max().item(), int(bT.argmax()),
                                             bT.max().item())
    assert bI[-1] < bt and bT[-1] < bt, (label, mode, "last block", bI[-1].item(), bT[-1].item())
    assert all(e < bt for e in row_errs), (label, mode, "rows", list(rows), row_errs)


def _fused(I, T, tau, mode):
    """The fused step through autograd (mae_clip_b200.clip_contrastive_loss): statistics, row loss and gradient in the
    forward call, the gradient form chosen on the device."""
    import mae_clip_b200 as m
    Ic, Tc = I.cuda().requires_grad_(True), T.cuda().requires_grad_(True)
    loss = m.clip_contrastive_loss(Ic, Tc, tau, mode=mode)
    loss.backward()
    return loss.item(), Ic.grad, Tc.grad


def _gate(I, T, tau, mode):
    """The gradient form the device picks for this batch (1 stored weights, 0 own rows), from one gated phased run of
    the stored form over every row - the fused step decides on the same finalized flags.  Returns (gate, loss, dI, dT)."""
    out = _phases_sharded(I.cuda(), T.cuda(), tau, mode, I.shape[0], stored=True, gated=True)
    return (_phases_sharded.last_gate,) + out[:3]


# ------------------------------------------------------------------ ragged batches at the large-tile size
RAGGED = [(4097, 256), (4223, 256), (4225, 256), (4351, 256), (8191, 256), (4097, 128), (4351, 128)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("scale", [1.0, 0.25])
@pytest.mark.parametrize("B,D", RAGGED)
def test_ragged_batch_fused_step(B, D, scale, mode):
    """B mod 128 in {1, 127} and B mod 256 on both sides of 128: a last row block, column tile, 256-row block of
    rowgrad_kernel / colgrad_kernel and column split that are partly padding.  Concentrated soft targets run the
    stored-weights form (gate 1), soft ones the own-rows sweep (gate 0); the gated phased run of the same batch is
    checked too."""
    I, T = _layernorm_batch(B, D, scale, seed=B % 97)
    ref = _oracle(("ln", B, D, scale), I, T, 1.0)
    gate, l2, dI2, dT2 = _gate(I, T, 1.0, mode)
    assert gate == (1 if scale == 1.0 else 0)
    # LayerNorm rows: the statistics span ~51 binades at 4096 rows, 61 at 8191 (the extreme rows drift apart)
    assert _exp_path(ref[3]) == ("wide" if (B, scale) == (8191, 1.0) else "fast")
    _check(f"ragged B={B} D={D} x{scale} phased", mode, l2, dI2, dT2, ref)
    _check(f"ragged B={B} D={D} x{scale} fused", mode, *_fused(I, T, 1.0, mode), ref)


def test_ragged_batch_host_entry():
    """B = 16500 through the host-buffer entry: the gradient runs in two strips of 65 and 64 row blocks, so the strip
    edge (row 8320) is not on a 256-row boundary and the last strip ends in a ragged block."""
    import ctypes
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    B, D, mode = 16500, 256, "tc_f16x3"
    I, T = _layernorm_batch(B, D, 1.0, seed=7)
    ref = _oracle(("ln", B, D, 1.0), I, T, 1.0)
    Ih, Th = I.pin_memory(), T.pin_memory()
    dI, dT = torch.full_like(Ih, float("nan")).pin_memory(), torch.full_like(Th, float("nan")).pin_memory()
    loss = torch.zeros(1).pin_memory()
    n = lib.mc_clip_loss_host_workspace_bytes(B, D, _lib.GEMM_MODES[mode])
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    _lib.check(lib.mc_clip_loss_fwd_bwd_host(Ih.data_ptr(), Th.data_ptr(), B, D, 1.0, _lib.GEMM_MODES[mode], loss.data_ptr(),
                                             dI.data_ptr(), dT.data_ptr(), ws.data_ptr(), n,
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
               "mc_clip_loss_fwd_bwd_host")
    assert _gate(I, T, 1.0, mode)[0] == 1
    _check(f"host entry B={B}", mode, loss.item(), dI, dT, ref, rows=range(8320 - 64, 8320 + 64))


# ------------------------------------------------------------------ far-negative row statistics
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [1000, 4133, 8191])
def test_cone_with_opposite_captions(B, mode):
    """Rows 0-2 have r ~ -50: 2^(-r log2 e) times the gradient weight scale overflows fp16 unless the padded columns
    of the ragged last tile get weight zero (they meet zero rows of the other tower: inf x 0 = NaN).  The statistics
    span ~200 binades, so the wide-range exponentials run.  B = 1000 takes pair_kernel's own-rows sweep, 4133 and 8191
    the large-tile kernels with the stored-weights form."""
    I, T = _cone_batch(B)
    ref = _oracle(("cone", B), I, T, 1.0)
    assert _span_binades(ref[3]) > FAST_PATH_BINADES + 8
    assert ref[3]["row_lse_s"][:3].max().item() < -30
    if B * B >= 4096 * 4096:
        gate, l2, dI2, dT2 = _gate(I, T, 1.0, mode)
        assert gate == 1
        _check(f"cone B={B} phased", mode, l2, dI2, dT2, ref, rows=(0, 1, 2))
    _check(f"cone B={B} fused", mode, *_fused(I, T, 1.0, mode), ref, rows=(0, 1, 2))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [1000, 4133])
def test_cone_with_opposite_images_own_rows(B, mode):
    """The transposed batch (three images opposite a cone of captions: column LSE c ~ -50) through the own-rows sweep
    of pair_kernel without tile flags, whose wide-range path forms e^(S_ji - c_i) q_i for the transposed strip."""
    I, T = _cone_batch(B, opposite_images=True)
    ref = _oracle(("cone-t", B), I, T, 1.0)
    assert _span_binades(ref[3]) > FAST_PATH_BINADES + 8
    assert ref[3]["col_lse_s"][:3].max().item() < -30
    loss, dI, dT, _ = _phases(I.cuda(), T.cuda(), 1.0, mode, sparse=False)
    _check(f"cone-t B={B} own rows", mode, loss, dI, dT, ref, rows=(0, 1, 2))


# ------------------------------------------------------------------ temperatures
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("scale,tau", [(1.0, 2.0), (0.7, 0.5)])
@pytest.mark.parametrize("B", [8192, 4223])
def test_temperature(B, scale, tau, mode):
    """tau != 1 at the large-tile sizes (max |S| = 128 and 250, inside the precision envelope of
    test_gradient_error_grows_with_the_logit_magnitude): the fused step, the sharded stored-weights form forced and
    gated (4096-row shards, or the whole ragged batch) and the length-B statistics of the column-partials sweep."""
    I, T = _layernorm_batch(B, 256, scale, seed=3)
    ref = _oracle(("ln", B, 256, scale), I, T, tau)
    st = ref[3]
    assert _exp_path(st) == "fast"
    Ic, Tc = I.cuda(), T.cuda()
    shard = 4096 if B % 128 == 0 else B
    for gated in (False, True):
        loss, dI, dT, _flags = _phases_sharded(Ic, Tc, tau, mode, shard, colpart=True, stored=True, gated=gated)
        assert _phases_sharded.last_gate == 1
        _check(f"tau={tau} x{scale} B={B} stored{' gated' if gated else ''}", mode, loss, dI, dT, ref)
        got = _phases_sharded.last_stats
        t_lse, t_gq = STAT_TOLS[mode]
        for k in ("row_lse_s", "col_lse_s", "row_lse_z"):
            assert rel_err(got[k], st[k]) < t_lse, (k, rel_err(got[k], st[k]))
        for k in ("row_g", "col_sum_p"):
            assert rel_err(got[k], st[k]) < t_gq, (k, rel_err(got[k], st[k]))
    _check(f"tau={tau} x{scale} B={B} fused", mode, *_fused(I, T, tau, mode), ref)


# ------------------------------------------------------------------ wide-range exponential path
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [4096, 4223])
def test_wide_range_path_at_large_size(B, mode):
    """Statistics spanning far more than 60 binades switch every gradient kernel to its separate per-column constants
    (wscale_kernel clears the fast flag): the forced stored-weights form (rowgrad_kernel's wide-range branch, kBwdP on
    the flagged tiles; and kBwdW without flags) and the fused step, whose gate takes the own-rows sweep here (rows of
    small norm have soft targets over every tile)."""
    I, T = _wide_norm_batch(B)
    ref = _oracle(("wide", B), I, T, 1.0)
    assert _span_binades(ref[3]) > FAST_PATH_BINADES + 8
    Ic, Tc = I.cuda(), T.cuda()
    for use_flags in (True, False):
        loss, dI, dT, _flags = _phases_sharded(Ic, Tc, 1.0, mode, B, stored=True, use_flags=use_flags)
        assert _phases_sharded.last_gate == 0
        _check(f"wide B={B} stored{'' if use_flags else ' noflags'}", mode, loss, dI, dT, ref)
    _check(f"wide B={B} fused", mode, *_fused(I, T, 1.0, mode), ref)


# ------------------------------------------------------------------ upstream gradient
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("form", ["stored", "stored_gated", "own_rows"])
@pytest.mark.parametrize("B", [8192, 4223])
def test_grad_loss_through_phased_forms(B, form, mode):
    """d(loss) = 0.37 as a device scalar through the phased gradient entry points (mc_clip_bwd_rows + mc_clip_bwd_cols,
    mc_clip_bwd), against the oracle's gradients for the same upstream gradient."""
    I, T = _layernorm_batch(B, 256, 1.0, seed=11)
    ref = _oracle(("ln", B, 256, 1.0), I, T, 1.0, grad_loss=0.37)
    shard = 4096 if B % 128 == 0 else B
    Ic, Tc = I.cuda(), T.cuda()
    if form == "own_rows":
        # mc_clip_bwd over every row WITH tile flags picks the gradient form itself (the stored one here): the ragged
        # batch runs it without flags, which is pair_kernel's own-rows sweep over every tile
        loss, dI, dT, _flags = _phases_sharded(Ic, Tc, 1.0, mode, shard, use_flags=shard != B, grad_loss=0.37)
    else:
        loss, dI, dT, _flags = _phases_sharded(Ic, Tc, 1.0, mode, shard, stored=True, gated=form == "stored_gated",
                                               grad_loss=0.37)
        assert _phases_sharded.last_gate == 1
    _check(f"grad_loss B={B} {form}", mode, loss, dI, dT, ref)
