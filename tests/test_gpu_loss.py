"""GPU parity of the contrastive soft-target loss and the standalone cross_entropy (rows L3-L6 of
SURVEY.md section 8) against the golden fixtures of the unmodified reference, the CPU oracle on
seeded inputs, and size-independent properties at the BASELINE sizes.

Tolerances (BASELINE.json north_star): fp32 engines - loss 1e-4 relative, gradients 1e-3 relative
(||d - ref|| / ||ref||); the single-pass half-precision engine is looser and says so below."""
import ctypes

import numpy as np
import pytest
import torch

from _loss_phases import _phases, _phases_sharded
from conftest import rel_err
from oracle import loss_ref

pytestmark = pytest.mark.gpu

LOSS_TOL, GRAD_TOL = 1e-4, 1e-3
# single-pass 16-bit operand engine: stated looser tolerance
LOOSE_LOSS_TOL, LOOSE_GRAD_TOL = 5e-4, 5e-3

FP32_MODES = ["simt_fp32", "tc_f16x3"]
ALL_MODES = FP32_MODES + ["tc_f16"]
CASES = ["b8_default", "b48_soft_tau05", "b33_dup_tau2", "b130_soft", "b64_verysoft"]


def _tols(mode):
    return (LOOSE_LOSS_TOL, LOOSE_GRAD_TOL) if mode == "tc_f16" else (LOSS_TOL, GRAD_TOL)


def _run(I, T, tau, mode, grad_scale=1.0):
    import mae_clip_b200 as m
    Ic = torch.as_tensor(I).cuda().requires_grad_(True)
    Tc = torch.as_tensor(T).cuda().requires_grad_(True)
    loss = m.clip_contrastive_loss(Ic, Tc, tau, mode=mode)
    (loss * grad_scale).backward()
    return loss.detach().cpu(), Ic.grad.cpu(), Tc.grad.cpu()


@pytest.mark.parametrize("mode", ALL_MODES)
@pytest.mark.parametrize("case", CASES)
def test_loss_golden(golden, case, mode):
    z = golden("clip_loss")
    tau = float(z[f"{case}.tau"])
    loss, dI, dT = _run(z[f"{case}.I"], z[f"{case}.T"], tau, mode)
    lt, gt = _tols(mode)
    ref = float(z[f"{case}.ref_loss_f64"])
    assert abs(loss.item() - ref) <= lt * abs(ref)
    assert rel_err(dI, z[f"{case}.ref_dI_f32"]) < gt
    assert rel_err(dT, z[f"{case}.ref_dT_f32"]) < gt


@pytest.mark.parametrize("mode", ALL_MODES)
@pytest.mark.parametrize("B,scale,tau", [(1, 1.0, 1.0), (2, 1.0, 1.0), (127, 0.1, 1.0), (256, 0.1, 2.0),
                                         (1024, 1.0, 1.0), (1024, 0.25, 0.5), (1000, 0.08, 1.0)])
def test_loss_vs_oracle_seeded(B, scale, tau, mode):
    """C2 shape (B=1024, D=256) and ragged / tiny batches against the fp64 closed form."""
    I = loss_ref.make_embeddings(B, 256, seed=0, scale=scale)
    T = loss_ref.make_embeddings(B, 256, seed=1, scale=scale)
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), tau, grad_loss=0.5)
    loss, dI, dT = _run(I, T, tau, mode, grad_scale=0.5)
    lt, gt = _tols(mode)
    assert abs(loss.item() - ref_loss) <= lt * max(abs(ref_loss), 1.0)  # B=1: the loss is exactly 0
    if np.linalg.norm(ref_dI) > 0:
        assert rel_err(dI, ref_dI) < gt
        assert rel_err(dT, ref_dT) < gt


@pytest.mark.parametrize("mode", ALL_MODES)
def test_loss_wide_norm_spread(mode):
    """Rows of very different norms: the row/column statistics span hundreds of binades, which
    switches the gradient sweep from its factored-exponential path to the six-exponential one."""
    B = 384
    g = torch.Generator().manual_seed(5)
    w = torch.logspace(-1.3, 0.0, B)[torch.randperm(B, generator=g)].unsqueeze(1)
    I = loss_ref.make_embeddings(B, 256, seed=12, scale=1.0) * w
    T = loss_ref.make_embeddings(B, 256, seed=13, scale=1.0) * w
    ref_loss, ref_dI, ref_dT, stats = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), 1.0)
    assert (stats["row_lse_z"].max() - stats["row_lse_z"].min()) * 1.4427 > 60
    loss, dI, dT = _run(I, T, 1.0, mode)
    lt, gt = _tols(mode)
    assert abs(loss.item() - ref_loss) <= lt * abs(ref_loss)
    assert rel_err(dI, ref_dI) < gt and rel_err(dT, ref_dT) < gt


@pytest.mark.parametrize("mode", FP32_MODES)
def test_loss_other_dims(mode):
    """D is a constructor argument of the heads (modules.py:59): not only 256."""
    for D in (64, 128, 512):
        I = loss_ref.make_embeddings(96, D, seed=3, scale=0.2)
        T = loss_ref.make_embeddings(96, D, seed=4, scale=0.2)
        ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), 1.0)
        loss, dI, dT = _run(I, T, 1.0, mode)
        assert abs(loss.item() - ref_loss) <= LOSS_TOL * abs(ref_loss)
        assert rel_err(dI, ref_dI) < GRAD_TOL and rel_err(dT, ref_dT) < GRAD_TOL


@pytest.mark.parametrize("mode", FP32_MODES)
def test_loss_properties_large(mode):
    """B=4096 (per-GPU shard size of C4), where the CPU oracle is slow: engine-vs-engine agreement
    plus properties - permutation equivariance of the gradients and invariance of the loss, and
    the directional derivative against a finite difference of the kernel's own loss."""
    import mae_clip_b200 as m
    B = 4096
    I = loss_ref.make_embeddings(B, 256, seed=7, scale=0.12)
    T = loss_ref.make_embeddings(B, 256, seed=8, scale=0.12)
    loss, dI, dT = _run(I, T, 1.0, mode)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0))
    loss_p, dI_p, dT_p = _run(I[perm], T[perm], 1.0, mode)
    assert abs(loss_p.item() - loss.item()) < 2e-5 * abs(loss.item())
    assert rel_err(dI_p, dI[perm]) < 1e-3 and rel_err(dT_p, dT[perm]) < 1e-3
    # directional derivative: (L(x + h v) - L(x - h v)) / 2h  vs  <grad, v>
    g = torch.Generator().manual_seed(1)
    vI, vT = torch.randn(B, 256, generator=g), torch.randn(B, 256, generator=g)
    vI, vT = vI / vI.norm(), vT / vT.norm()
    h = 0.05
    with torch.no_grad():
        lp = m.clip_contrastive_loss((I + h * vI).cuda(), (T + h * vT).cuda(), 1.0, mode=mode).item()
        lm = m.clip_contrastive_loss((I - h * vI).cuda(), (T - h * vT).cuda(), 1.0, mode=mode).item()
    fd = (lp - lm) / (2 * h)
    an = (dI * vI).sum().item() + (dT * vT).sum().item()
    assert abs(fd - an) < 5e-2 * max(abs(an), 1e-4) + 1e-5
    if mode != "simt_fp32":
        l0, dI0, dT0 = _run(I, T, 1.0, "simt_fp32")
        assert abs(loss.item() - l0.item()) < LOSS_TOL * abs(l0.item())
        assert rel_err(dI, dI0) < GRAD_TOL and rel_err(dT, dT0) < GRAD_TOL


def test_loss_no_grad_and_eval():
    import mae_clip_b200 as m
    I = loss_ref.make_embeddings(64, 256, seed=0).cuda()
    T = loss_ref.make_embeddings(64, 256, seed=1).cuda()
    with torch.no_grad():
        l0 = m.clip_contrastive_loss(I, T, 1.0)
    assert l0.grad_fn is None
    ref = loss_ref.clip_loss_ref(I.cpu(), T.cpu(), 1.0)
    assert abs(l0.item() - ref.item()) < LOSS_TOL * abs(ref.item())


def test_loss_host_buffer_entry_point():
    """mc_clip_loss_fwd_bwd_host: the e2e call of bench.py (host buffers in, loss + grads out)."""
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    B, D = 256, 256
    I = loss_ref.make_embeddings(B, D, seed=0, scale=0.1).pin_memory()
    T = loss_ref.make_embeddings(B, D, seed=1, scale=0.1).pin_memory()
    dI, dT = torch.empty_like(I).pin_memory(), torch.empty_like(T).pin_memory()
    loss = torch.zeros(1).pin_memory()
    for mode in (0, 1):
        n = lib.mc_clip_loss_host_workspace_bytes(B, D, mode)
        ws = torch.empty(n, dtype=torch.uint8, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.mc_clip_loss_fwd_bwd_host(I.data_ptr(), T.data_ptr(), B, D, 1.0, mode, loss.data_ptr(),
                                                 dI.data_ptr(), dT.data_ptr(), ws.data_ptr(), n,
                                                 ctypes.c_void_p(st)))
        ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), 1.0)
        assert abs(loss.item() - ref_loss) < LOSS_TOL * abs(ref_loss)
        assert rel_err(dI, ref_dI) < GRAD_TOL and rel_err(dT, ref_dT) < GRAD_TOL


@pytest.mark.parametrize("B", [16384, 16500, 32768])
def test_loss_host_entry_strips_match_single_sweep(B, monkeypatch):
    """From B = 16384 the host-buffer entry runs the gradient sweep in two row strips and copies a strip
    back while the next is swept: same loss and gradients as the device-resident single sweep, ragged last strip
    included, and identical on a second call (events / copy stream reused correctly)."""
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    D, mode = 256, 1
    monkeypatch.setenv("MAE_CLIP_HOST_CHUNKS", "1")   # the inbound side has its own test; same operand scale here
    I = loss_ref.make_embeddings(B, D, seed=3).pin_memory()
    T = (0.6 * I + 0.8 * loss_ref.make_embeddings(B, D, seed=4)).pin_memory()   # correlated pairs: a real diagonal
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = lib.mc_clip_loss_fused_workspace_bytes(B, D, mode)
    ws0 = torch.empty(n0, dtype=torch.uint8, device="cuda")
    Id, Td = I.cuda(), T.cuda()
    l0, dI0, dT0 = torch.zeros(1, device="cuda"), torch.empty_like(Id), torch.empty_like(Td)
    _lib.check(lib.mc_clip_loss_fwd_bwd(Id.data_ptr(), Td.data_ptr(), B, D, 1.0, mode, l0.data_ptr(), dI0.data_ptr(),
                                        dT0.data_ptr(), ws0.data_ptr(), n0, st), "mc_clip_loss_fwd_bwd")
    n = lib.mc_clip_loss_host_workspace_bytes(B, D, mode)
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    outs = []
    for _ in range(2):
        dI, dT = torch.full_like(I, float("nan")).pin_memory(), torch.full_like(T, float("nan")).pin_memory()
        loss = torch.zeros(1).pin_memory()
        _lib.check(lib.mc_clip_loss_fwd_bwd_host(I.data_ptr(), T.data_ptr(), B, D, 1.0, mode, loss.data_ptr(),
                                                 dI.data_ptr(), dT.data_ptr(), ws.data_ptr(), n, st),
                   "mc_clip_loss_fwd_bwd_host")
        outs.append((loss.clone(), dI.clone(), dT.clone()))
    loss, dI, dT = outs[0]
    assert torch.isfinite(dI).all() and torch.isfinite(dT).all()
    assert abs(loss.item() - l0.item()) <= 1e-6 * abs(l0.item())
    assert rel_err(dI, dI0.cpu()) < 1e-5 and rel_err(dT, dT0.cpu()) < 1e-5
    assert torch.equal(outs[1][1], dI) and torch.equal(outs[1][2], dT) and torch.equal(outs[1][0], loss)


@pytest.mark.parametrize("chunks", [1, 2, 4, 8])
@pytest.mark.parametrize("B,scale", [(8192, 1.0), (16384, 1.0), (8192, 0.25)])
def test_loss_host_entry_chunked_inbound_copy(B, scale, chunks, monkeypatch):
    """The host-buffer entry stages the batch and runs the statistics sweep chunk by chunk behind the inbound copy
    (MAE_CLIP_HOST_CHUNKS row chunks, arrival-ordered launches of the sweep): every chunk count meets the parity bar
    against the fp64 blockwise oracle - LayerNorm-scale rows (diagonal tile flags) and the soft regime (x 0.25: every
    tile flagged) - and stays close to the device-resident step.  (The chunked form fixes the operand scale from the
    first chunk with a binade of headroom, so the fp16 hi/lo planes differ from the resident step's in the last bit of
    the lo plane; the fp16 rounding of the gradient weights turns that into ~1e-4 between two results that are each
    ~3e-4 from fp64.)"""
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    D, mode = 256, 1
    Id, Td, (ref_loss, ref_dI, ref_dT, _stats) = _c4_batch_and_oracle(B, scale)
    I, T = Id.cpu().pin_memory(), Td.cpu().pin_memory()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = lib.mc_clip_loss_fused_workspace_bytes(B, D, mode)
    ws0 = torch.empty(n0, dtype=torch.uint8, device="cuda")
    l0, dI0, dT0 = torch.zeros(1, device="cuda"), torch.empty_like(Id), torch.empty_like(Td)
    _lib.check(lib.mc_clip_loss_fwd_bwd(Id.data_ptr(), Td.data_ptr(), B, D, 1.0, mode, l0.data_ptr(), dI0.data_ptr(),
                                        dT0.data_ptr(), ws0.data_ptr(), n0, st), "mc_clip_loss_fwd_bwd")
    monkeypatch.setenv("MAE_CLIP_HOST_CHUNKS", str(chunks))
    n = lib.mc_clip_loss_host_workspace_bytes(B, D, mode)
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        dI, dT = torch.full_like(I, float("nan")).pin_memory(), torch.full_like(T, float("nan")).pin_memory()
        loss = torch.zeros(1).pin_memory()
        _lib.check(lib.mc_clip_loss_fwd_bwd_host(I.data_ptr(), T.data_ptr(), B, D, 1.0, mode, loss.data_ptr(),
                                                 dI.data_ptr(), dT.data_ptr(), ws.data_ptr(), n, st),
                   "mc_clip_loss_fwd_bwd_host")
        assert torch.isfinite(dI).all() and torch.isfinite(dT).all()
        assert abs(loss.item() - ref_loss) <= LOSS_TOL * abs(ref_loss)
        eI, eT = rel_err(dI, ref_dI), rel_err(dT, ref_dT)
        assert eI < GRAD_TOL and eT < GRAD_TOL, (eI, eT)
        assert abs(loss.item() - l0.item()) <= 1e-5 * abs(l0.item())
        assert rel_err(dI, dI0.cpu()) < 5e-4 and rel_err(dT, dT0.cpu()) < 5e-4


def test_loss_host_entry_chunked_scale_outgrown(monkeypatch, capfd):
    """Rows of a later chunk exceed the headroom of the first chunk's scale: the device-side check trips and the
    step is redone from the resident copy - the caller sees the plain result."""
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    B, D, mode = 8192, 256, 1
    I = loss_ref.make_embeddings(B, D, seed=7)
    T = 0.6 * I + 0.8 * loss_ref.make_embeddings(B, D, seed=8)
    monkeypatch.setenv("MAE_CLIP_HOST_CHUNKS", "4")
    I[: B // 4] *= 0.2          # chunk 0 is small: the later rows are 5x its maximum
    T[: B // 4] *= 0.2
    I, T = I.pin_memory(), T.pin_memory()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = lib.mc_clip_loss_fused_workspace_bytes(B, D, mode)
    ws0 = torch.empty(n0, dtype=torch.uint8, device="cuda")
    Id, Td = I.cuda(), T.cuda()
    l0, dI0, dT0 = torch.zeros(1, device="cuda"), torch.empty_like(Id), torch.empty_like(Td)
    _lib.check(lib.mc_clip_loss_fwd_bwd(Id.data_ptr(), Td.data_ptr(), B, D, 1.0, mode, l0.data_ptr(), dI0.data_ptr(),
                                        dT0.data_ptr(), ws0.data_ptr(), n0, st), "mc_clip_loss_fwd_bwd")
    n = lib.mc_clip_loss_host_workspace_bytes(B, D, mode)
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    dI, dT = torch.full_like(I, float("nan")).pin_memory(), torch.full_like(T, float("nan")).pin_memory()
    loss = torch.zeros(1).pin_memory()
    monkeypatch.setenv("MAE_CLIP_HOST_TRACE", "1")      # the library prints its timeline: shows which path ran
    capfd.readouterr()
    _lib.check(lib.mc_clip_loss_fwd_bwd_host(I.data_ptr(), T.data_ptr(), B, D, 1.0, mode, loss.data_ptr(),
                                             dI.data_ptr(), dT.data_ptr(), ws.data_ptr(), n, st),
               "mc_clip_loss_fwd_bwd_host")
    err = capfd.readouterr().err
    assert "staged[1]" in err and err.rstrip().splitlines()[-1].endswith("end")     # chunked attempt ...
    assert any(line.endswith(" staged") for line in err.splitlines())                # ... then the plain redo
    assert abs(loss.item() - l0.item()) <= 1e-6 * abs(l0.item())
    assert rel_err(dI, dI0.cpu()) < 1e-5 and rel_err(dT, dT0.cpu()) < 1e-5


def test_abi_error_codes():
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    x = torch.zeros(16, 256, device="cuda")
    out = torch.zeros(1, device="cuda")
    ws = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    rc = lib.mc_clip_loss_fwd_bwd(x.data_ptr(), x.data_ptr(), 16, 256, 1.0, 0, out.data_ptr(), None, None,
                                  ws.data_ptr(), 16, None)
    assert rc == 5 and b"workspace" in lib.mc_last_error_string()
    rc = lib.mc_clip_loss_fwd_bwd(None, x.data_ptr(), 16, 256, 1.0, 0, out.data_ptr(), None, None,
                                  ws.data_ptr(), 1024, None)
    assert rc == 1
    rc = lib.mc_clip_loss_fwd_bwd(x.data_ptr(), x.data_ptr(), 16, 256, -1.0, 0, out.data_ptr(), None, None,
                                  ws.data_ptr(), 1024, None)
    assert rc == 1
    assert lib.mc_device_supported(0) == 1


def test_abi_error_codes_next_rows_and_peer():
    """Bad arguments come back as status codes with a message, never as a crash or an exception across the ABI."""
    import ctypes as C
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    x = torch.zeros(64, 256, device="cuda")
    i64 = torch.zeros(64, dtype=torch.int64, device="cuda")
    ws = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    tab = (C.c_void_p * 1)(x.data_ptr())
    n1 = (C.c_int64 * 1)(64 * 256)
    # AdamW: step counts from 1; betas inside [0, 1)
    assert lib.mc_adamw_step(1, tab, tab, tab, tab, n1, 1e-3, 0.9, 0.999, 1e-8, 0.0, 0, None, None) == 1
    assert b"step" in lib.mc_last_error_string()
    assert lib.mc_adamw_step(1, tab, tab, tab, tab, n1, 1e-3, 1.5, 0.999, 1e-8, 0.0, 1, None, None) == 1
    assert lib.mc_adamw_step(0, None, None, None, None, None, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, None, None) == 0  # empty: fine
    # retrieval: k beyond the bank, k beyond the shared-memory limit, short workspace
    assert lib.mc_similarity_topk(p(x), 1, p(x), 64, 256, 65, p(x), p(i64), None, p(ws), ws.numel(), None) == 1
    assert lib.mc_similarity_topk(p(x), 1, p(x), 64, 256, 2000, p(x), p(i64), None, p(ws), ws.numel(), None) in (1, 6)
    assert lib.mc_similarity_topk(p(x), 1, p(x), 64, 256, 4, p(x), p(i64), None, p(ws), 8, None) == 5
    # peer primitives: world outside [1, 16], rank outside the world, null epoch counter
    assert lib.mc_peer_barrier(tab, 0, 17, p(ws), 1.0, None) == 1
    assert lib.mc_peer_barrier(tab, 3, 1, p(ws), 1.0, None) == 1
    assert lib.mc_peer_barrier(tab, 0, 1, None, 1.0, None) == 1
    assert lib.mc_peer_publish(p(x), 0, 4, 4, tab, 4, 0, 1, None) == 1
    # peer staging feeds the tcgen05 engines only
    assert lib.mc_clip_prepare_peers(tab, tab, 1, 64, 256, 0, p(ws), p(ws), None) == 6
    # data feed: zero std
    m3, s3 = (C.c_float * 3)(0.5, 0.5, 0.5), (C.c_float * 3)(0.5, 0.0, 0.5)
    u8 = torch.zeros(1, 4, 4, 3, dtype=torch.uint8, device="cuda")
    assert lib.mc_normalize_images(p(u8), 1, 4, 4, m3, s3, 255.0, p(x), None) == 1
    # restore_tokens backward: rows must be 16-byte multiples
    assert lib.mc_restore_tokens_bwd(p(x), 4, 0, p(i64), 1, 8, 3, 4, p(x), p(x), p(ws), ws.numel(), None) == 6
    torch.cuda.synchronize()  # nothing above may have launched a faulting kernel


# ------------------------------------------------------------------ cross_entropy (CLIP.py:46-52)
def test_cross_entropy_golden(golden):
    import mae_clip_b200 as m
    z = golden("cross_entropy")
    p, t = torch.from_numpy(z["rect.preds"]).cuda(), torch.from_numpy(z["rect.targets"]).cuda()
    np.testing.assert_allclose(m.cross_entropy(p, t, reduction="none").cpu().numpy(), z["rect.ref_none"], rtol=2e-6,
                               atol=1e-6)
    np.testing.assert_allclose(m.cross_entropy(p, t, reduction="mean").cpu().numpy(), z["rect.ref_mean"], rtol=2e-6)
    assert m.cross_entropy(p, t, reduction="sum") is None
    sp = torch.from_numpy(z["sq.preds"]).cuda().requires_grad_(True)
    st = torch.from_numpy(z["sq.targets"]).cuda().requires_grad_(True)
    out = m.cross_entropy(sp.T, st.T, reduction="none")  # transposed views, as CLIP.py:41
    np.testing.assert_allclose(out.detach().cpu().numpy(), z["sq.ref_none_T"], rtol=2e-6, atol=1e-6)
    (out * torch.from_numpy(z["sq.w"]).cuda()).sum().backward()
    np.testing.assert_allclose(sp.grad.cpu().numpy(), z["sq.ref_dpreds_T"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(st.grad.cpu().numpy(), z["sq.ref_dtargets_T"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("rows,cols", [(1, 1), (3, 5), (257, 1023), (1024, 1024), (100, 4097), (260, 1000),
                                       (4096, 333), (36, 130)])
@pytest.mark.parametrize("transposed", [False, True])
def test_cross_entropy_vs_oracle(rows, cols, transposed):
    import mae_clip_b200 as m
    g = torch.Generator().manual_seed(rows * 7 + cols)
    shape = (cols, rows) if transposed else (rows, cols)
    p0 = torch.randn(shape, generator=g) * 4
    t0 = torch.rand(shape, generator=g)
    w = torch.rand(rows, generator=g)

    def run(dev, fn):
        p = p0.detach().clone().to(dev).requires_grad_(True)
        t = t0.detach().clone().to(dev).requires_grad_(True)
        pv, tv = (p.T, t.T) if transposed else (p, t)
        out = fn(pv, tv, "none")
        (out * w.to(dev)).sum().backward()
        return out.detach().cpu(), p.grad.cpu(), t.grad.cpu()

    o_ref, dp_ref, dt_ref = run("cpu", loss_ref.soft_cross_entropy_ref)
    o, dp, dt = run("cuda", m.cross_entropy)
    assert rel_err(o, o_ref) < 1e-5 and rel_err(dp, dp_ref) < 1e-5 and rel_err(dt, dt_ref) < 1e-5


def test_cross_entropy_empty_rows():
    import mae_clip_b200 as m
    out = m.cross_entropy(torch.zeros(0, 5, device="cuda"), torch.zeros(0, 5, device="cuda"))
    assert out.shape == (0,)


# ------------------------------------------------------------------ tile flags (soft-target sparsity)
@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
def test_tile_flags_skip_only_what_is_negligible(mode):
    """LayerNorm-scale rows: Z_ii = 256 towers over every other Z_ij, so only the diagonal tiles carry soft-target
    mass - the flagged sweeps must reproduce the dense ones (the dropped terms are below 2^-44) and the oracle."""
    B = 1024 + 128
    I = loss_ref.make_embeddings(B, 256, seed=21, scale=1.0).cuda()
    T = loss_ref.make_embeddings(B, 256, seed=22, scale=1.0).cuda()
    ld, dId, dTd, _ = _phases(I, T, 1.0, mode, sparse=False)
    ls, dIs, dTs, flags = _phases(I, T, 1.0, mode, sparse=True)
    assert torch.equal(flags, torch.eye(flags.shape[0], dtype=torch.uint8))       # diagonal tiles only
    assert abs(ls - ld) <= 1e-6 * abs(ld)
    # flagged and dense gradients come from different kernels (split: the softmax and soft-target parts of the weights
    # are rounded to fp16 separately; dense: together): a few 1e-5 of fp16 weight rounding, both ~2.5e-4 from fp64
    assert rel_err(dIs, dId) < 5e-5 and rel_err(dTs, dTd) < 5e-5
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.cpu().numpy(), T.cpu().numpy(), 1.0)
    lt, gt = _tols(mode)
    assert abs(ls - ref_loss) <= lt * abs(ref_loss)
    assert rel_err(dIs, ref_dI) < gt and rel_err(dTs, ref_dT) < gt


def test_tile_flags_soft_regime_keeps_every_tile():
    """Small norms: every Z_ij is within a few units of Z_ii, all tiles matter, nothing may be skipped."""
    B = 640
    I = loss_ref.make_embeddings(B, 256, seed=31, scale=0.1).cuda()
    T = loss_ref.make_embeddings(B, 256, seed=32, scale=0.1).cuda()
    ls, dIs, dTs, flags = _phases(I, T, 1.0, "tc_f16x3", sparse=True)
    assert bool(flags.all())
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.cpu().numpy(), T.cpu().numpy(), 1.0)
    assert abs(ls - ref_loss) <= LOSS_TOL * abs(ref_loss)
    assert rel_err(dIs, ref_dI) < GRAD_TOL and rel_err(dTs, ref_dT) < GRAD_TOL


def test_tile_flags_find_duplicates_across_tiles():
    """Near-duplicate samples in different tiles share their soft-target mass (P_ij ~ 1/2): the off-diagonal tile
    pair must be flagged (both orientations, through the transpose in mc_clip_flags_finalize) and the gradients
    must match the oracle - a skipped tile there would be a visible error."""
    B = 768
    I0 = loss_ref.make_embeddings(B, 256, seed=41, scale=1.0)
    T0 = loss_ref.make_embeddings(B, 256, seed=42, scale=1.0)
    I0[700], T0[700] = I0[3], T0[3]                     # row 700 (tile 5) duplicates row 3 (tile 0)
    I0[300] = I0[200] * 0.999                           # near-duplicate images only (tiles 2 and 1)
    I, T = I0.cuda(), T0.cuda()
    ls, dIs, dTs, flags = _phases(I, T, 1.0, "tc_f16x3", sparse=True)
    assert flags[0, 5] == 1 and flags[5, 0] == 1
    assert flags.sum().item() < flags.numel()           # still sparse elsewhere
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I0.numpy(), T0.numpy(), 1.0)
    assert abs(ls - ref_loss) <= LOSS_TOL * abs(ref_loss)
    assert rel_err(dIs, ref_dI) < GRAD_TOL and rel_err(dTs, ref_dT) < GRAD_TOL
    ld, dId, dTd, _ = _phases(I, T, 1.0, "tc_f16x3", sparse=False)
    assert rel_err(dIs, dId) < 1e-5 and rel_err(dTs, dTd) < 1e-5


@pytest.mark.parametrize("B", [640 + 64, 4096, 4096 + 128])
@pytest.mark.parametrize("scale,tau", [(1.0, 1.0), (0.5, 1.0), (0.35, 1.0), (0.6, 0.25), (0.1, 1.0)])
def test_tile_flags_are_a_superset_of_the_exact_relevance(scale, tau, B):
    """The engine's flags come from a bound (probe Z against Z_ii); the oracle computes the exact set of tiles holding
    a P_ij or P_ji >= 2^-44 in fp64.  Flags must cover it in every regime (hard, intermediate, soft), with a few rows
    of larger norm thrown in so that rz_i > Z_ii for the others.  B = 704 runs the probe of pair_kernel<kStats>; from
    4096 on rowsweep_kernel<kRsZ> (tiles on or above the diagonal, row criterion + column criterion against the smallest
    Z_jj of the tile) - 4224 is not a multiple of 256."""
    I0 = loss_ref.make_embeddings(B, 256, seed=51, scale=scale)
    T0 = loss_ref.make_embeddings(B, 256, seed=52, scale=scale)
    I0[5] *= 1.3; T0[400] *= 1.2; I0[401] = I0[17]          # norm outliers and a cross-tile duplicate
    _ls, _dI, _dT, flags = _phases(I0.cuda(), T0.cuda(), tau, "tc_f16x3", sparse=True)
    exact = torch.from_numpy(loss_ref.tile_relevance(I0.numpy(), T0.numpy(), tau))
    assert flags.shape == exact.shape
    assert bool((flags.bool() | ~exact).all()), "a tile with soft-target mass was not flagged"
    if scale == 1.0:
        assert flags.sum().item() <= exact.sum().item() + 4   # and the bound is tight in the hard regime


@pytest.mark.parametrize("B", [4096, 4096 + 128])
def test_tile_flags_partial_probe_falls_back_to_the_full_probe(B):
    """rowsweep_kernel<kRsZ> multiplies out only the leading 128 dimensions of each tower and bounds the rest of Z_ij by
    Cauchy-Schwarz (clip_loss_tc.cu, probe_chunks).  Rows whose leading dimensions are EMPTY make that bound useless
    (it equals Z_ii for every pair): the partial probe flags every tile, the device-side verdict (probe_gate_kernel)
    clears the bitmap and the full probe runs - the result must be the diagonal again, and the step must match the oracle."""
    I0 = loss_ref.make_embeddings(B, 256, seed=71, scale=1.0)
    T0 = loss_ref.make_embeddings(B, 256, seed=72, scale=1.0)
    I0[:, :128] = 0.0
    T0[:, :128] = 0.0
    I0 *= 16.0 / I0.norm(dim=1, keepdim=True)           # back to the LayerNorm norm: Z_ii = 256, off-diagonal sigma 16
    T0 *= 16.0 / T0.norm(dim=1, keepdim=True)
    ls, dIs, dTs, flags = _phases(I0.cuda(), T0.cuda(), 1.0, "tc_f16x3", sparse=True)
    nt = flags.shape[0]
    # the diagonal (plus, at most, a borderline pair): nowhere near the all-ones bitmap of the partial probe
    assert bool(torch.diagonal(flags).all()) and flags.sum().item() <= nt + 4
    exact = torch.from_numpy(loss_ref.tile_relevance(I0.numpy(), T0.numpy(), 1.0))
    assert bool((flags.bool() | ~exact).all())
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I0.numpy(), T0.numpy(), 1.0)
    assert abs(ls - ref_loss) <= LOSS_TOL * abs(ref_loss)
    assert rel_err(dIs, ref_dI) < GRAD_TOL and rel_err(dTs, ref_dT) < GRAD_TOL


def test_tile_flags_partial_probe_falls_back_per_row_shard():
    """The same batch under row sharding (4096-row strips of B = 8192, the size from which a strip runs rowsweep_kernel):
    every strip takes its own verdict and re-probes; flags and gradients must equal the single call's."""
    B = 8192
    I0 = loss_ref.make_embeddings(B, 256, seed=73, scale=1.0)
    T0 = loss_ref.make_embeddings(B, 256, seed=74, scale=1.0)
    I0[:, :128] = 0.0
    T0[:, :128] = 0.0
    I0 *= 16.0 / I0.norm(dim=1, keepdim=True)           # back to the LayerNorm norm: Z_ii = 256, off-diagonal sigma 16
    T0 *= 16.0 / T0.norm(dim=1, keepdim=True)
    Ic, Tc = I0.cuda(), T0.cuda()
    l1, dI1, dT1, single = _phases(Ic, Tc, 1.0, "tc_f16x3", sparse=True)
    nt = single.shape[0]
    assert bool(torch.diagonal(single).all()) and single.sum().item() <= nt + 8
    l2, dI2, dT2, sharded = _phases_sharded(Ic, Tc, 1.0, "tc_f16x3", 4096, colpart=True)
    sharded = sharded.cpu()
    assert bool(torch.diagonal(sharded).all()) and sharded.sum().item() <= nt + 8
    assert abs(l1 - l2) <= 1e-6 * abs(l1)
    assert rel_err(dI2.cpu(), dI1) < 5e-5 and rel_err(dT2.cpu(), dT1) < 5e-5


@pytest.mark.parametrize("scale", [1.0, 0.45])
def test_tile_flags_of_row_shards_cover_the_single_call_flags(scale):
    """Under row sharding rowsweep_kernel<kRsZ> probes every tile of the strip with the row criterion only (the raw flags
    of a strip also drive its exact-Z statistics, so they must be complete per rank); after mc_clip_flags_finalize (which
    ORs the transposed relation over all shards) the bitmap must cover what the single call (upper triangle, row + column
    criteria) flags - which the test above pins on the exact fp64 relevance.  Near-duplicates far apart included."""
    B = 8192
    I = loss_ref.make_embeddings(B, 256, seed=61, scale=scale)
    T = loss_ref.make_embeddings(B, 256, seed=62, scale=scale)
    I[7000] = I[100]; T[7000] = T[100]; I[4200] = I[4100]; T[130] = T[8000]       # cross-tile near-duplicates
    Ic, Tc = I.cuda(), T.cuda()
    _l, _dI, _dT, single = _phases(Ic, Tc, 1.0, "tc_f16x3", sparse=True)
    for b in (2048, 4096):
        _l2, _dI2, _dT2, sharded = _phases_sharded(Ic, Tc, 1.0, "tc_f16x3", b, colpart=True)
        assert sharded.shape == single.shape
        assert bool((sharded.cpu().bool() | ~single.cpu().bool()).all()), "a tile flagged by the single call is missing under sharding"
        if scale == 1.0:
            assert sharded.sum().item() <= single.sum().item() + 8


# ------------------------------------------------------------------ parity AT the benchmarked size (BASELINE config 4)
_C4_CACHE = {}


def _c4_batch_and_oracle(B, scale):
    """bench.py's C4 batch (4096-row blocks of LayerNorm'd gaussian rows, seeds 1000 + k / 5000 + k) and its fp64
    blockwise oracle (``oracle/loss_blockwise.py``, plain torch float64 ON THE GPU as the checker - never the product)."""
    from oracle import loss_blockwise
    key = (B, scale)
    if key not in _C4_CACHE:
        _C4_CACHE.clear()   # one batch resident at a time
        blk = 4096
        I = torch.cat([loss_ref.make_embeddings(blk, 256, seed=1000 + k, scale=scale) for k in range(B // blk)]).cuda()
        T = torch.cat([loss_ref.make_embeddings(blk, 256, seed=5000 + k, scale=scale) for k in range(B // blk)]).cuda()
        ref = loss_blockwise.clip_loss_blockwise_f64(I, T, 1.0, rows=1024)
        _C4_CACHE[key] = (I, T, ref)
    return _C4_CACHE[key]


@pytest.mark.parametrize("variant", ["fused_flags", "dense", "shards4096_flags", "shards4096_colpart", "shards4096_stored",
                                     "shards4096_stored_noflags", "shards4096_stored_gated", "host_entry"])
@pytest.mark.parametrize("B", [8192, 32768])
def test_loss_c4_size_vs_fp64_blockwise(B, variant):
    """The benchmarked path - B = 32768 (and 8192), D = 256, LayerNorm-scale rows (tile-flag density 1/256), probe +
    exact-Z statistics, 4096-row shards, the strip-wise host entry - against the fp64 oracle at its own size:
    loss <= 1e-4, gradients <= 1e-3 relative (north_star), for the fp32-class engine with tile flags on AND off."""
    import ctypes as C
    from mae_clip_b200 import _lib
    I, T, (ref_loss, ref_dI, ref_dT, _stats) = _c4_batch_and_oracle(B, 1.0)
    if variant == "fused_flags":
        lib = _lib.lib()
        n = lib.mc_clip_loss_fused_workspace_bytes(B, 256, 1)
        ws = torch.empty(n, dtype=torch.uint8, device="cuda")
        l, dI, dT = torch.zeros(1, device="cuda"), torch.empty_like(I), torch.empty_like(T)
        _lib.check(lib.mc_clip_loss_fwd_bwd(I.data_ptr(), T.data_ptr(), B, 256, 1.0, 1, l.data_ptr(), dI.data_ptr(),
                                            dT.data_ptr(), ws.data_ptr(), n, _lib.cur_stream()))
        loss = l.item()
    elif variant == "dense":
        loss, dI, dT, _ = _phases(I, T, 1.0, "tc_f16x3", sparse=False)
    elif variant.startswith("shards4096"):
        loss, dI, dT, flags = _phases_sharded(I, T, 1.0, "tc_f16x3", 4096, colpart="flags" not in variant,
                                              stored="stored" in variant, use_flags=not variant.endswith("noflags"),
                                              gated=variant.endswith("gated"))
        if variant.endswith("gated"):
            assert _phases_sharded.last_gate == 1     # concentrated soft targets: the stored form ran
        assert flags.float().mean().item() < 0.02      # the sparse path is what ran (diagonal tiles + a few neighbours)
    else:
        lib = _lib.lib()
        Ih, Th = I.cpu().pin_memory(), T.cpu().pin_memory()
        dI, dT = torch.empty_like(Ih).pin_memory(), torch.empty_like(Th).pin_memory()
        l = torch.zeros(1).pin_memory()
        n = lib.mc_clip_loss_host_workspace_bytes(B, 256, 1)
        ws = torch.empty(n, dtype=torch.uint8, device="cuda")
        _lib.check(lib.mc_clip_loss_fwd_bwd_host(Ih.data_ptr(), Th.data_ptr(), B, 256, 1.0, 1, l.data_ptr(), dI.data_ptr(),
                                                 dT.data_ptr(), ws.data_ptr(), n, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        loss = l.item()
    assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss), (loss, ref_loss)
    eI, eT = rel_err(dI, ref_dI), rel_err(dT, ref_dT)
    print(f"c4 parity B={B} {variant}: loss rel {abs(loss - ref_loss) / abs(ref_loss):.2e}, dI {eI:.2e}, dT {eT:.2e}")
    assert eI < GRAD_TOL and eT < GRAD_TOL, (eI, eT)


@pytest.mark.parametrize("B", [8192, 32768])
def test_loss_c4_size_single_pass_engine_vs_fp64_blockwise(B):
    """Same check for the single-pass fp16 engine at ITS stated tolerance (5e-4 / 5e-3)."""
    I, T, (ref_loss, ref_dI, ref_dT, _stats) = _c4_batch_and_oracle(B, 1.0)
    loss, dI, dT, _ = _phases(I, T, 1.0, "tc_f16", sparse=True)
    assert abs(loss - ref_loss) <= LOOSE_LOSS_TOL * abs(ref_loss)
    assert rel_err(dI, ref_dI) < LOOSE_GRAD_TOL and rel_err(dT, ref_dT) < LOOSE_GRAD_TOL


def test_loss_c4_size_soft_regime_vs_fp64_blockwise():
    """B = 8192 with embeddings x 0.25 (every tile carries soft-target mass: flag density 1.0, the regime bench.py
    reports as `roofline.soft`): flagged and dense sweeps against the fp64 oracle."""
    B = 8192
    I, T, (ref_loss, ref_dI, ref_dT, _stats) = _c4_batch_and_oracle(B, 0.25)
    for sparse in (True, False):
        loss, dI, dT, flags = _phases(I, T, 1.0, "tc_f16x3", sparse=sparse)
        if sparse:
            assert bool(flags.all())
        assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss)
        assert rel_err(dI, ref_dI) < GRAD_TOL and rel_err(dT, ref_dT) < GRAD_TOL
    # row shards with the device-side choice of the gradient form: every tile is flagged, so the gate picks the own-rows
    # sweep (0) and the stored-weights kernels return at once; forced stored form (no gate) for the same batch
    for gated in (True, False):
        loss, dI, dT, flags = _phases_sharded(I, T, 1.0, "tc_f16x3", 4096, colpart=True, stored=True, gated=gated)
        if gated:
            assert _phases_sharded.last_gate == 0
        assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss)
        assert rel_err(dI, ref_dI) < GRAD_TOL and rel_err(dT, ref_dT) < GRAD_TOL


@pytest.mark.parametrize("scale", [1.0, 0.25])
@pytest.mark.parametrize("B,b", [(1152, 384), (1280, 1280), (640, 128)])
def test_stored_weights_gradient_small_and_ragged_shapes(B, b, scale):
    """mc_clip_bwd_rows / mc_clip_bwd_cols called directly at sizes below the automatic switch (4096 x 4096 logits), where
    the padded shapes matter: B not a multiple of 256 (rowgrad_kernel's row blocks and colgrad_kernel's column blocks are
    256 wide), strips of 128 - 1280 rows, concentrated and soft targets - against the closed-form fp64 oracle."""
    I = loss_ref.make_embeddings(B, 256, seed=31, scale=scale).cuda()
    T = loss_ref.make_embeddings(B, 256, seed=32, scale=scale).cuda()
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.cpu().numpy(), T.cpu().numpy(), 1.0)
    for gated in (False, True):
        loss, dI, dT, _flags = _phases_sharded(I, T, 1.0, "tc_f16x3", b, colpart=True, stored=True, gated=gated)
        assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss)
        assert rel_err(dI, ref_dI) < GRAD_TOL and rel_err(dT, ref_dT) < GRAD_TOL, (gated, rel_err(dI, ref_dI), rel_err(dT, ref_dT))


@pytest.mark.parametrize("B,D,scale", [(4096, 128, 1.0), (4096, 256, 1.0), (4224, 128, 0.3)])
def test_large_tile_kernels_at_their_smallest_size(B, D, scale):
    """From 4096 x 4096 logits on the fused step runs rowsweep_kernel (statistics) and rowgrad_kernel + colgrad_kernel
    (stored-weights gradient): both embedding widths of the tcgen05 engine, a batch that is not a multiple of 256, and
    a batch whose soft targets are not concentrated (the device-side gate then takes the own-rows sweep) against the
    closed-form fp64 oracle."""
    import mae_clip_b200 as m
    I = loss_ref.make_embeddings(B, D, seed=41, scale=scale)
    T = loss_ref.make_embeddings(B, D, seed=42, scale=scale)
    Ic, Tc = I.cuda().requires_grad_(True), T.cuda().requires_grad_(True)
    loss = m.clip_contrastive_loss(Ic, Tc, 1.0, mode="tc_f16x3")
    loss.backward()
    ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I.numpy(), T.numpy(), 1.0)
    assert abs(loss.item() - ref_loss) <= LOSS_TOL * abs(ref_loss)
    assert rel_err(Ic.grad, ref_dI) < GRAD_TOL and rel_err(Tc.grad, ref_dT) < GRAD_TOL


def test_fused_step_is_bit_deterministic():
    """No atomics on floats anywhere in the path (every partial is folded in a fixed order): repeated calls on the same
    inputs give the same bits - also a cheap detector of races in the kernels' mbarrier protocols (tools/
    stress_determinism.py runs the long version)."""
    from mae_clip_b200 import _lib
    from mae_clip_b200._lib import check, cur_stream, ptr
    lib = _lib.lib()
    B, D = 8192, 256
    I = loss_ref.make_embeddings(B, D, seed=71).cuda()
    T = loss_ref.make_embeddings(B, D, seed=72).cuda()
    for mode in (1, 2):
        n = lib.mc_clip_loss_fused_workspace_bytes(B, D, mode)
        ws = torch.zeros(n, dtype=torch.uint8, device="cuda")
        loss, dI, dT = torch.zeros(1, device="cuda"), torch.empty_like(I), torch.empty_like(T)
        ref = None
        for _ in range(12):
            dI.fill_(float("nan")); dT.fill_(float("nan"))
            check(lib.mc_clip_loss_fwd_bwd(ptr(I), ptr(T), B, D, 1.0, mode, ptr(loss), ptr(dI), ptr(dT), ptr(ws), n, cur_stream()))
            cur = (loss.clone(), dI.clone(), dT.clone())
            if ref is None:
                ref = cur
            assert all(torch.equal(a, b) for a, b in zip(ref, cur))


@pytest.mark.parametrize("B", [2048, 4096])
def test_gradient_error_grows_with_the_logit_magnitude(B):
    """The fp32-class engine's remaining error is the tensor core's truncating fp32 accumulation, proportional to the size
    of the logits: rows of norm 16 (what the reference's LayerNorm emits) give ~2.7e-4 on the gradients, norm 24 ~6.5e-4,
    norm 32 ~2.1e-3 - the last one is OUTSIDE the 1e-3 bar and is pinned here so that the limit stays documented
    (DESIGN 4.1 "Precision"); the loss itself stays at 1e-6 throughout.  Same numbers on the small-problem kernels
    (B = 2048) and the large-tile ones (B = 4096)."""
    import mae_clip_b200 as m
    from oracle import loss_blockwise
    for scale, bound in ((1.0, 1e-3), (1.5, 1e-3), (2.0, 4e-3)):
        I = loss_ref.make_embeddings(B, 256, seed=81, scale=scale).cuda()
        T = loss_ref.make_embeddings(B, 256, seed=82, scale=scale).cuda()
        ref_loss, ref_dI, ref_dT, _ = loss_blockwise.clip_loss_blockwise_f64(I, T, 1.0, rows=1024)
        Ic, Tc = I.clone().requires_grad_(True), T.clone().requires_grad_(True)
        loss = m.clip_contrastive_loss(Ic, Tc, 1.0, mode="tc_f16x3")
        loss.backward()
        assert abs(loss.item() - ref_loss) <= 1e-5 * abs(ref_loss)
        assert rel_err(Ic.grad, ref_dI) < bound and rel_err(Tc.grad, ref_dT) < bound, (scale, rel_err(Ic.grad, ref_dI))


# ------------------------------------------------------------------ autograd plumbing (round-1 advisor findings)
def test_fp32_fma_engine_state_survives_other_ops_between_forward_and_backward():
    """The fp32 FMA engine keeps its S / S^T / Z strips from the statistics sweep to the gradient sweep.  Through the
    row-sharded Function (mae_clip_b200/dist.py) that state lives in the autograd context, not in the shared scratch
    cache: other mae_clip_b200 ops between forward and backward, and a second backward over a retained graph, must not
    change the gradients.  D = 64 also covers the automatic fall-back of the tcgen05 modes to this engine."""
    import mae_clip_b200 as m
    from mae_clip_b200.dist import global_clip_loss
    for mode, D in (("simt_fp32", 256), ("tc_f16x3", 64)):
        B = 192
        I0 = loss_ref.make_embeddings(B, D, seed=71, scale=0.2)
        T0 = loss_ref.make_embeddings(B, D, seed=72, scale=0.2)
        I, T = I0.cuda().requires_grad_(True), T0.cuda().requires_grad_(True)
        loss = global_clip_loss(I, T, 1.0, mode=mode)
        # other work that goes through the same per-stream scratch buffer
        J = loss_ref.make_embeddings(320, D, seed=73, scale=0.3).cuda().requires_grad_(True)
        m.clip_contrastive_loss(J, J * 0.5, 1.0, mode="simt_fp32").backward()
        global_clip_loss(J.detach(), J.detach() * 0.5, 1.0, mode=mode)
        pred = torch.randn(4, 196, 768, device="cuda", requires_grad=True)
        m.masked_mse_loss(pred, torch.randn(4, 3, 224, 224, device="cuda"), torch.ones(4, 196, device="cuda")).backward()
        loss.backward(retain_graph=True)
        g1 = (I.grad.clone(), T.grad.clone())
        I.grad = T.grad = None
        loss.backward()
        ref_loss, ref_dI, ref_dT, _ = loss_ref.clip_loss_closed_form(I0.numpy(), T0.numpy(), 1.0)
        assert abs(loss.item() - ref_loss) <= LOSS_TOL * abs(ref_loss)
        assert rel_err(g1[0], ref_dI) < GRAD_TOL and rel_err(g1[1], ref_dT) < GRAD_TOL
        assert torch.equal(I.grad, g1[0]) and torch.equal(T.grad, g1[1])


def test_no_grad_forward_does_not_run_the_gradient_sweep():
    """`main.py:115` evaluates under torch.no_grad() with parameters that require grad: the loss and the heads must not
    run (or allocate for) their backward there."""
    import mae_clip_b200 as m
    from mae_clip_b200 import _lib
    lib = _lib.lib()
    I = loss_ref.make_embeddings(256, 256, seed=0).cuda().requires_grad_(True)
    T = loss_ref.make_embeddings(256, 256, seed=1).cuda().requires_grad_(True)
    n0 = lib.mc_kernel_launch_count()
    l_grad = m.clip_contrastive_loss(I, T, 1.0)
    n1 = lib.mc_kernel_launch_count()
    with torch.no_grad():
        l_eval = m.clip_contrastive_loss(I, T, 1.0)
    n2 = lib.mc_kernel_launch_count()
    assert l_eval.grad_fn is None and l_eval.item() == l_grad.item()
    assert n2 - n1 < n1 - n0       # no gradient sweep / finalize launches
    head = m.ProjectionHead(512).cuda().train()
    x = torch.randn(64, 512, device="cuda", requires_grad=True)
    keep = torch.ones(64, 256, dtype=torch.uint8, device="cuda")
    with torch.no_grad():
        out = head(x, keep_mask=keep)
    assert out.grad_fn is None


@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
@pytest.mark.parametrize("B,shard,scale", [(640, 128, 0.1), (1000, 1000, 0.3), (768, 384, 1.0), (129, 129, 0.5),
                                           (4096, 4096, 1.0), (4096 + 128, 4096 + 128, 1.0)])
def test_column_partials_statistics_match_oracle(B, shard, scale, mode):
    """Column LSE of S from the per-warp column partials (no transposed strip): ragged batches, a strip that is the
    whole batch, strips of one row block, rows of very different scale in one column (exponentials are taken against
    each column's OWN maximum, so nothing underflows) - the five statistic vectors against the fp64 closed form.
    From 4096 rows on the sweep is rowsweep_kernel<kRsS>: its 32 x 32 blocks share one set of exponentials between the
    row LSE and the column partials (weighted against the block maximum); the text row scaled by 6 puts logits of
    +-300 next to +-50 in its blocks, so columns there fall out of the safe range and take the kernel's exact path."""
    from mae_clip_b200 import _lib
    from mae_clip_b200._lib import check, cur_stream, ptr
    lib = _lib.lib()
    md = _lib.GEMM_MODES[mode]
    g = torch.Generator().manual_seed(B)
    I0 = loss_ref.make_embeddings(B, 256, seed=81, scale=scale)
    T0 = loss_ref.make_embeddings(B, 256, seed=82, scale=scale)
    I0[1] *= 6.0; T0[B // 2] *= 6.0; I0[B - 1] *= 0.01          # a column far above and one far below the others
    I, T = I0.cuda(), T0.cuda()
    _l, _dI, _dT, stats = loss_ref.clip_loss_closed_form(I0.numpy(), T0.numpy(), 1.0)
    planes = torch.empty(lib.mc_clip_planes_bytes(B, 256, md), dtype=torch.uint8, device="cuda")
    check(lib.mc_clip_prepare(ptr(I), ptr(T), B, B, 256, 0, md, ptr(planes), cur_stream()))
    W = (B + shard - 1) // shard
    if B % shard or shard % 128:
        W, shard = 1, B                       # row offsets must be multiples of 128: one strip = the whole batch
    ws = torch.empty(lib.mc_clip_stats_colpart_workspace_bytes(shard, B, 256, md), dtype=torch.uint8, device="cuda")
    r, rz, ps = torch.empty(B, device="cuda"), torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
    cparts = torch.empty(W, B, device="cuda")
    for k in range(W):
        o = k * shard
        check(lib.mc_clip_stats_colpart(ptr(planes), shard, B, 256, o, 1.0, md, ptr(r[o:]), ptr(cparts[k]), ptr(rz[o:]), ptr(ps[o:]),
                                        None, ptr(ws), ws.numel(), cur_stream()))
    c = torch.empty(B, device="cuda")
    check(lib.mc_clip_colpart_merge(ptr(cparts), W, B, B, ptr(c), cur_stream()))
    tol = 2e-5 if mode == "tc_f16x3" else 2e-3
    assert rel_err(c, stats["col_lse_s"]) < tol
    assert rel_err(r, stats["row_lse_s"]) < tol and rel_err(rz, stats["row_lse_z"]) < tol
