"""The phased forms of the contrastive loss step through the C ABI on one GPU (test infrastructure).

``_phases`` runs the whole batch as one call per phase (prepare -> statistics -> flags finalize -> row loss ->
gradient); ``_phases_sharded`` runs the row-sharded form that the ranks of a multi-GPU job use
(``mae_clip_b200/dist.py``), back to back on one device.  Both are shared by the loss test modules."""
import torch


def _grad_loss_ptr(grad_loss, dev):
    """A device scalar holding ``grad_loss`` (the upstream gradient of the loss) and its pointer; None: no scaling."""
    from mae_clip_b200._lib import ptr
    if grad_loss is None:
        return None, None
    g = torch.full((1,), float(grad_loss), device=dev)
    return g, ptr(g)


def _phases(I, T, tau, mode, sparse, grad_loss=None):
    """prepare -> stats -> (flags finalize) -> rowloss -> bwd through the C ABI on one GPU; returns loss, dI, dT, flags.
    ``grad_loss``: upstream gradient of the loss, passed to the gradient sweep as a device scalar."""
    from mae_clip_b200 import _lib
    from mae_clip_b200._lib import check, cur_stream, ptr
    lib = _lib.lib()
    md = _lib.GEMM_MODES[mode]
    B, D = I.shape
    dev = I.device
    planes = torch.empty(lib.mc_clip_planes_bytes(B, D, md), dtype=torch.uint8, device=dev)
    ws = torch.empty(lib.mc_clip_loss_workspace_bytes(B, B, D, md), dtype=torch.uint8, device=dev)
    st4 = torch.empty(4, B, device=dev)
    gq = torch.empty(2, B, device=dev)
    loss = torch.empty(1, device=dev)
    dI, dT = torch.empty_like(I), torch.empty_like(T)
    nf = lib.mc_clip_tile_flags_bytes(B, B, D, md) if sparse else 0
    raw = torch.empty(nf, dtype=torch.uint8, device=dev) if nf else None
    fin = torch.empty(nf, dtype=torch.uint8, device=dev) if nf else None
    _gl, gl = _grad_loss_ptr(grad_loss, dev)
    s = cur_stream()
    check(lib.mc_clip_prepare(ptr(I), ptr(T), B, B, D, 0, md, ptr(planes), s))
    check(lib.mc_clip_stats(ptr(I), ptr(T), ptr(planes), B, B, D, 0, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]), ptr(st4[3]),
                            ptr(raw), ptr(ws), ws.numel(), s))
    if nf:
        check(lib.mc_clip_flags_finalize(ptr(raw), B, B, 0, ptr(fin), s))
    check(lib.mc_clip_rowloss(ptr(I), ptr(T), ptr(planes), B, B, D, 0, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]), ptr(st4[3]),
                              ptr(gq[0]), ptr(gq[1]), ptr(loss), ptr(fin), ptr(ws), ws.numel(), s))
    check(lib.mc_clip_bwd(ptr(I), ptr(T), ptr(planes), B, B, D, 0, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]), ptr(gq[0]),
                          ptr(gq[1]), gl, ptr(dI), ptr(dT), ptr(fin), ptr(ws), ws.numel(), s))
    torch.cuda.synchronize()
    nt = (B + 127) // 128
    return loss.item(), dI.cpu(), dT.cpu(), (fin.cpu().reshape(nt, nt) if nf else None)


def _phases_sharded(I, T, tau, mode, shard_rows, colpart=False, stored=False, use_flags=True, gated=False, grad_loss=None):
    """The row-sharded form of the step (what the ranks of a multi-GPU job run, mae_clip_b200/dist.py) back to back on
    one GPU: every shard of `shard_rows` rows runs its own statistics / row-loss / gradient sweeps with a row offset,
    the length-B vectors and the tile-flag bitmap are assembled in between exactly as the exchange steps do.

    Shards are whole 128-row blocks; a batch that is not a multiple of 128 runs as one shard of all B rows (row offset
    0), which is how the fused single-GPU step calls the stored-weights halves.  ``grad_loss``: upstream gradient of the
    loss, passed to the gradient sweeps as a device scalar.  Afterwards ``_phases_sharded.last_gate`` holds the device's
    choice of the gradient form for the finalized flags (1 = stored weights, 0 = own rows; None without the stored form)
    and ``_phases_sharded.last_stats`` the length-B statistics vectors, keyed as the oracles key them."""
    from mae_clip_b200 import _lib
    from mae_clip_b200._lib import check, cur_stream, ptr
    lib = _lib.lib()
    md = _lib.GEMM_MODES[mode]
    B, D = I.shape
    b = shard_rows
    assert B % b == 0 and (b % 128 == 0 or b == B), (B, b)
    W = B // b
    nt = (B + 127) // 128
    dev = I.device
    s = cur_stream()
    _gl, gl = _grad_loss_ptr(grad_loss, dev)
    planes = torch.empty(lib.mc_clip_planes_bytes(B, D, md), dtype=torch.uint8, device=dev)
    ws = torch.empty(lib.mc_clip_loss_workspace_bytes(b, B, D, md), dtype=torch.uint8, device=dev)
    nf = lib.mc_clip_tile_flags_bytes(b, B, D, md)
    st4 = torch.empty(4, B, device=dev)
    gq = torch.empty(2, B, device=dev)
    parts = torch.empty(W, device=dev)
    raw_all = torch.empty(W * nf, dtype=torch.uint8, device=dev)
    fin = torch.empty(W, nf, dtype=torch.uint8, device=dev)
    dI, dT = torch.empty_like(I), torch.empty_like(T)
    check(lib.mc_clip_prepare(ptr(I), ptr(T), B, B, D, 0, md, ptr(planes), s))
    if colpart:
        # the column-partials form: every shard returns LSE over ITS rows of every column; the vectors are merged as
        # the ranks do after exchanging them (mae_clip_b200/dist.py PeerStep)
        ws = torch.empty(max(ws.numel(), lib.mc_clip_stats_colpart_workspace_bytes(b, B, D, md)), dtype=torch.uint8, device=dev)
        cparts = torch.empty(W, B, device=dev)
    for k in range(W):
        o = k * b
        if colpart:
            check(lib.mc_clip_stats_colpart(ptr(planes), b, B, D, o, tau, md, ptr(st4[0, o:]), ptr(cparts[k]), ptr(st4[2, o:]),
                                            ptr(st4[3, o:]), ptr(raw_all[k * nf:]), ptr(ws), ws.numel(), s))
        else:
            check(lib.mc_clip_stats(ptr(I), ptr(T), ptr(planes), b, B, D, o, tau, md, ptr(st4[0, o:]), ptr(st4[1, o:]),
                                    ptr(st4[2, o:]), ptr(st4[3, o:]), ptr(raw_all[k * nf:]), ptr(ws), ws.numel(), s))
    if colpart:
        check(lib.mc_clip_colpart_merge(ptr(cparts), W, B, B, ptr(st4[1]), s))
    for k in range(W):
        check(lib.mc_clip_flags_finalize(ptr(raw_all), B, b, k * b, ptr(fin[k]), s))
    for k in range(W):
        o = k * b
        check(lib.mc_clip_rowloss(ptr(I), ptr(T), ptr(planes), b, B, D, o, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]),
                                  ptr(st4[3, o:]), ptr(gq[0, o:]), ptr(gq[1, o:]), ptr(parts[k:]), ptr(fin[k]), ptr(ws),
                                  ws.numel(), s))
    _phases_sharded.last_gate = None
    if stored:
        # the stored-weights form as the ranks run it (dist.PeerStep): per shard the row half (dT, the fp16 weight strip,
        # the soft-target part of the shard's dI) and the column half over EVERY row of dI; the shards' partial dI are
        # then summed (the peer reduce)
        Wbuf = torch.empty(lib.mc_clip_stored_weights_bytes(b, B), dtype=torch.uint8, device=dev)
        wsc = torch.empty(lib.mc_clip_bwd_cols_workspace_bytes(B, D), dtype=torch.uint8, device=dev)
        Bp = nt * 128
        # the form (stored / own rows) the device chooses from the density of the whole flag bitmap; a gated call
        # follows that choice, an ungated one runs the stored form whatever it says
        gate = torch.full((1,), -1, dtype=torch.int32, device=dev)
        check(lib.mc_clip_bwd_gate(ptr(fin), fin.numel(), ptr(gate), s), "mc_clip_bwd_gate")
        dI_sum = torch.zeros_like(dI)
        for k in range(W):
            o = k * b
            diz = torch.zeros(Bp, D, device=dev)
            part = torch.zeros(B, D, device=dev)
            check(lib.mc_clip_bwd_rows(ptr(planes), b, B, D, o, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]), ptr(gq[0]),
                                       ptr(gq[1]), gl, ptr(dT[o:]), ptr(diz[o:]), ptr(Wbuf), ptr(fin[k]) if use_flags else None,
                                       ptr(gate) if gated else None, ptr(dI[o:]) if gated else None, ptr(ws), ws.numel(), s),
                  "mc_clip_bwd_rows")
            check(lib.mc_clip_bwd_cols(ptr(planes), B, D, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]), ptr(gq[1]), gl,
                                       ptr(Wbuf), b, o, 0, B, ptr(diz), ptr(part), ptr(gate) if gated else None, ptr(wsc),
                                       wsc.numel(), s), "mc_clip_bwd_cols")
            dI_sum += part
        _phases_sharded.last_gate = gate.item()
        if not gated or _phases_sharded.last_gate == 1:
            dI = dI_sum       # the stored form ran: the shards' partial dI summed (the peer reduce)
    else:
        for k in range(W):
            o = k * b
            check(lib.mc_clip_bwd(ptr(I), ptr(T), ptr(planes), b, B, D, o, tau, md, ptr(st4[0]), ptr(st4[1]), ptr(st4[2]),
                                  ptr(gq[0]), ptr(gq[1]), gl, ptr(dI[o:]), ptr(dT[o:]), ptr(fin[k]) if use_flags else None, ptr(ws),
                                  ws.numel(), s))
    torch.cuda.synchronize()
    _phases_sharded.last_stats = {"row_lse_s": st4[0], "col_lse_s": st4[1], "row_lse_z": st4[2], "row_g": gq[0],
                                  "col_sum_p": gq[1]}
    return parts.sum().item(), dI, dT, fin.reshape(nt, -1)


_phases_sharded.last_gate = None
_phases_sharded.last_stats = None
