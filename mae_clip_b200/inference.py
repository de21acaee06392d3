"""Inference-side retrieval ("next" row 3, SURVEY.md section 8 f).

Mirrors ``/root/reference/inference.py:30-47`` (``find_matches``) without the tokenizer download and
the matplotlib display: L2-normalise both embedding sets, ``text @ image.T``, ``torch.topk(n * 5)``,
every fifth hit.  The arithmetic is one streaming pass over the image bank plus an exact radix
select (``mc_similarity_topk``); ties resolve to the lower index.

Retrieval evaluation (not in the reference): ``retrieval_ranks`` / ``retrieval_recall`` /
``evaluate_retrieval`` give the text->image and image->text ranks and recall@K of a whole validation
set from one tensor-core pass over the (Q, N) cosine scores, which are never stored
(``mc_retrieval_ranks``).

``retrieval_topk`` is the query-batch path: the exact top-k of those same tensor-core scores for every query, in
workspace that does not grow with queries x bank (``mc_retrieval_topk``).  ``similarity_topk`` stays the fp32-exact
path (and the only one for D > 256 or ``return_scores``).
"""
from __future__ import annotations

import torch

from ._lib import check, cur_stream, lib, ptr, require_cuda, workspace
from .functional import _mode


def similarity_topk(text_embeddings: torch.Tensor, image_embeddings: torch.Tensor, k: int, return_scores: bool = False):
    """(Q, D), (N, D) -> values (Q, k) fp32, indices (Q, k) int64 of the k most similar images per
    query by cosine similarity (``inference.py:42-46``).  ``return_scores`` also returns the (Q, N)
    similarity matrix (``dot_similarity``)."""
    require_cuda(text_embeddings, image_embeddings)
    t = text_embeddings.detach().float().contiguous()
    x = image_embeddings.detach().float().contiguous()
    if t.dim() != 2 or x.dim() != 2 or t.shape[1] != x.shape[1]:
        raise ValueError("similarity_topk expects (Q, D) text and (N, D) image embeddings")
    Q, D = t.shape
    N = x.shape[0]
    if k > N:
        raise RuntimeError(f"selected index k={k} out of range for {N} candidates")  # as torch.topk
    dev = x.device
    vals = torch.empty(Q, k, device=dev, dtype=torch.float32)
    idx = torch.empty(Q, k, device=dev, dtype=torch.int64)
    scores = torch.empty(Q, N, device=dev, dtype=torch.float32) if return_scores else None
    if Q == 0 or N == 0:
        return (vals, idx, scores) if return_scores else (vals, idx)
    with torch.cuda.device(dev):
        nws = lib().mc_similarity_topk_workspace_bytes(Q, N, D)
        ws = workspace(nws, dev)
        check(lib().mc_similarity_topk(ptr(t), Q, ptr(x), N, D, k, ptr(vals), ptr(idx), ptr(scores), ptr(ws), ws.numel(),
                                       cur_stream()), "mc_similarity_topk")
    return (vals, idx, scores) if return_scores else (vals, idx)


def get_image_embeddings(model, loader, device=None):
    """``inference.py:12-28`` minus checkpoint loading: image tower + projection over a loader, eval / no_grad."""
    device = device if device is not None else next(model.parameters()).device
    model.eval()
    out = []
    with torch.no_grad():
        for batch in loader:
            feats = model.image_encoder(batch["image"].to(device))
            out.append(model.image_projection(feats))
    return model, torch.cat(out)


def find_matches(model, image_embeddings, encoded_query, image_filenames, n=9):
    """``inference.py:30-47``: ``encoded_query`` is the tokenizer output for ONE query
    (``{"input_ids": ..., "attention_mask": ...}``, lists or tensors).  Returns the ``n`` matched
    file names (the reference then plots them)."""
    device = image_embeddings.device
    batch = {k: torch.as_tensor(v).to(device) for k, v in encoded_query.items() if k in ("input_ids", "attention_mask")}
    with torch.no_grad():
        text_features = model.text_encoder(input_ids=batch["input_ids"], attention_mask=batch["attention_mask"])
        text_embeddings = model.text_projection(text_features)
    _, indices = similarity_topk(text_embeddings[:1], image_embeddings, n * 5)
    return [image_filenames[i] for i in indices[0, ::5].tolist()]


def _ranks_launch(t, x, tti, mode):
    Q, D = t.shape
    N = x.shape[0]
    dev = x.device
    t2i = torch.empty(Q, device=dev, dtype=torch.int32)
    i2t = torch.empty(N, device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        nws = lib().mc_retrieval_ranks_workspace_bytes(Q, N, D, mode)
        ws = workspace(nws, dev)
        check(lib().mc_retrieval_ranks(ptr(t), Q, ptr(x), N, D, ptr(tti), mode, ptr(t2i), ptr(i2t), ptr(ws), ws.numel(),
                                       cur_stream()), "mc_retrieval_ranks")
    return t2i.long(), i2t.long()


def _embedding_pair(text_embeddings, image_embeddings, what):
    require_cuda(text_embeddings, image_embeddings)
    t = text_embeddings.detach().float().contiguous()
    x = image_embeddings.detach().float().contiguous()
    if t.dim() != 2 or x.dim() != 2 or t.shape[1] != x.shape[1]:
        raise ValueError(f"{what} expect (Q, D) text and (N, D) image embeddings with the same D, got "
                         f"{tuple(t.shape)} and {tuple(x.shape)}")
    if t.device != x.device:
        raise ValueError("text and image embeddings must be on the same device")
    return t, x


def _ranks_inputs(text_embeddings, image_embeddings, text_to_image):
    t, x = _embedding_pair(text_embeddings, image_embeddings, "retrieval ranks")
    Q, N = t.shape[0], x.shape[0]
    if text_to_image is None:
        if Q != N:
            raise ValueError(f"without text_to_image caption q pairs with image q, so Q ({Q}) must equal N ({N})")
        tti = None
    else:
        tti = torch.as_tensor(text_to_image).to(device=x.device, dtype=torch.int64).contiguous()
        if tti.shape != (Q,):
            raise ValueError(f"text_to_image must have shape ({Q},), got {tuple(tti.shape)}")
    return t, x, tti


def retrieval_ranks(text_embeddings: torch.Tensor, image_embeddings: torch.Tensor, text_to_image=None, mode=None):
    """Text->image and image->text ranks of a retrieval evaluation, from cosine similarities
    ``s[q, n] = <text_q / max(|text_q|, 1e-12), image_n / max(|image_n|, 1e-12)>`` (``inference.py:42-44``).

    ``text_embeddings`` (Q, D) and ``image_embeddings`` (N, D) on the device; ``text_to_image`` (Q,) int64 is the
    index of each caption's image (``None``: Q == N and caption q pairs with image q).  Returns int64 tensors
    ``(t2i_rank (Q,), i2t_rank (N,))``:

    * ``t2i_rank[q]`` = number of images n != g(q) with ``s[q, n] > s[q, g(q)]`` (0: the caption's own image first);
    * ``i2t_rank[n]`` = number of captions q with g(q) != n and ``s[q, n] > max_{q': g(q') = n} s[q', n]``, the rank
      of the image's best-ranked caption (COCO / Karpathy-split convention); -1 for an image without a caption.

    Comparisons are strict (exact ties favour the positive).  The counts are exact and identical run to run, but
    they compare the engine's scores: ``mode`` ``"tc_f16x3"`` (the package default, fp32-class) or ``"tc_f16"``
    (one fp16 pass); a candidate whose true score lies within 3e-5 (tc_f16x3) / 2e-3 (tc_f16), absolute, of the
    threshold may be counted on either side.  D <= 256 and D % 4 == 0.  The (Q, N) matrix is never stored.
    Checking ``text_to_image`` against [0, N) synchronises with the device once."""
    mode = _mode(mode)
    with torch.no_grad():
        t, x, tti = _ranks_inputs(text_embeddings, image_embeddings, text_to_image)
        Q, N = t.shape[0], x.shape[0]
        if tti is not None and Q > 0 and bool(((tti < 0) | (tti >= N)).any()):
            raise ValueError(f"text_to_image entries must lie in [0, {N})")
        if Q == 0 or N == 0:
            return (torch.zeros(Q, device=x.device, dtype=torch.int64),
                    torch.full((N,), -1, device=x.device, dtype=torch.int64))
        return _ranks_launch(t, x, tti, mode)


def retrieval_topk(text_embeddings: torch.Tensor, image_embeddings: torch.Tensor, k: int, mode=None):
    """(Q, D) queries, (N, D) bank -> values (Q, k) fp32, indices (Q, k) int64: the k best images of every query by
    the cosine score ``retrieval_ranks`` uses, computed on the tensor cores.

    The result is the exact top-k of the engine's scores: descending, exact ties to the lower index, identical run
    to run; the values are those scores, within 3e-5 (``mode`` ``"tc_f16x3"``, the package default) or 2e-3
    (``"tc_f16"``), absolute, of the true cosine.  Image-to-text top-k is the same call with the arguments swapped.
    The (Q, N) matrix is never stored: the workspace is O((Q + N) D + Q (k + C)) for a bank chunk C of at most
    65 536 (see ``mc_retrieval_topk`` in the header).  Limits: k <= N (``RuntimeError``, as ``torch.topk``),
    k <= 1024, D <= 256 and D % 4 == 0.  For D > 256 or the full score matrix use ``similarity_topk``."""
    mode = _mode(mode)
    with torch.no_grad():
        t, x = _embedding_pair(text_embeddings, image_embeddings, "retrieval_topk")
        Q, D = t.shape
        N = x.shape[0]
        if k < 0 or k > N:
            raise RuntimeError(f"selected index k={k} out of range for {N} candidates")  # as torch.topk
        if k > 1024:
            raise ValueError(f"retrieval_topk supports k <= 1024, got k={k}")
        if D > 256 or D % 4 != 0:
            raise ValueError(f"retrieval_topk needs D <= 256 and D % 4 == 0, got D={D} (similarity_topk takes any D)")
        dev = x.device
        vals = torch.empty(Q, k, device=dev, dtype=torch.float32)
        idx = torch.empty(Q, k, device=dev, dtype=torch.int64)
        if Q == 0 or k == 0:
            return vals, idx
        with torch.cuda.device(dev):
            nws = lib().mc_retrieval_topk_workspace_bytes(Q, N, D, k, mode)
            ws = workspace(nws, dev)
            check(lib().mc_retrieval_topk(ptr(t), Q, ptr(x), N, D, k, mode, ptr(vals), ptr(idx), ptr(ws), ws.numel(),
                                          cur_stream()), "mc_retrieval_topk")
        return vals, idx


def _recall_from_ranks(t2i, i2t, ks):
    """Device tensor of recall@K values: [t2i@k for k in ks] + [i2t@k for k in ks]."""
    kt = torch.as_tensor(list(ks), device=t2i.device, dtype=torch.int64)
    r_t = ((t2i[None, :] >= 0) & (t2i[None, :] < kt[:, None])).double().sum(1) / max(t2i.numel(), 1)
    has = (i2t >= 0)
    r_i = ((i2t[None, :] >= 0) & (i2t[None, :] < kt[:, None])).double().sum(1) / has.sum().clamp_min(1).double()
    r_i = torch.where(has.any(), r_i, torch.full_like(r_i, float("nan")))
    return torch.cat([r_t, r_i])


def retrieval_recall(text_embeddings: torch.Tensor, image_embeddings: torch.Tensor, text_to_image=None,
                     ks=(1, 5, 10), mode=None):
    """Recall@K in both directions: ``{"text_to_image_R@K": ..., "image_to_text_R@K": ...}`` (python floats), the
    fraction of captions / images with ``0 <= rank < K`` (ranks as ``retrieval_ranks`` defines them; images without
    a caption are left out of image->text recall).  Synchronises with the device once."""
    mode = _mode(mode)
    ks = [int(k) for k in ks]
    with torch.no_grad():
        t, x, tti = _ranks_inputs(text_embeddings, image_embeddings, text_to_image)
        Q, N = t.shape[0], x.shape[0]
        bad = torch.zeros((), device=x.device, dtype=torch.bool)
        if tti is not None and Q > 0:
            # checked together with the result (one transfer); the kernel reads a clamped copy meanwhile
            bad = ((tti < 0) | (tti >= N)).any()
            tti = tti.clamp(0, max(N - 1, 0))
        if Q == 0 or N == 0:
            t2i = torch.zeros(Q, device=x.device, dtype=torch.int64)
            i2t = torch.full((N,), -1, device=x.device, dtype=torch.int64)
        else:
            t2i, i2t = _ranks_launch(t, x, tti, mode)
        vals = torch.cat([bad.double()[None], _recall_from_ranks(t2i, i2t, ks)]).tolist()
    if vals[0]:
        raise ValueError(f"text_to_image entries must lie in [0, {N})")
    out = {}
    for j, k in enumerate(ks):
        out[f"text_to_image_R@{k}"] = vals[1 + j]
    for j, k in enumerate(ks):
        out[f"image_to_text_R@{k}"] = vals[1 + len(ks) + j]
    return out


def _embed_pairs(model, loader, device=None):
    """Image and text embeddings of every row of a reference-style loader (``image``, ``input_ids``,
    ``attention_mask``; one row per caption, as ``CLIPDataset`` yields them), in eval mode under no_grad.
    Returns ``(image_embeddings (R, P), text_embeddings (R, P))``; the model's train / eval mode is restored."""
    device = device if device is not None else next(model.parameters()).device
    was_training = model.training
    model.eval()
    imgs, txts = [], []
    try:
        with torch.no_grad():
            for batch in loader:
                imgs.append(model.image_projection(model.image_encoder(batch["image"].to(device))))
                txts.append(model.text_projection(model.text_encoder(
                    input_ids=batch["input_ids"].to(device), attention_mask=batch["attention_mask"].to(device))))
    finally:
        model.train(was_training)
    return torch.cat(imgs), torch.cat(txts)


def evaluate_retrieval(model, loader, ks=(1, 5, 10), image_ids=None, mode=None):
    """Recall@K of a CLIP model over a validation loader, in both directions (``retrieval_recall``).

    Every row of the loader is one (image, caption) pair.  ``image_ids`` (one id per row, in loader order) names the
    image of each row: rows with the same id share one image, embedded from its first row, so a COCO-style set with
    five captions per image is ranked against each image once.  Without ``image_ids`` the rows are one-to-one pairs."""
    image_emb, text_emb = _embed_pairs(model, loader)
    if image_ids is None:
        return retrieval_recall(text_emb, image_emb, None, ks=ks, mode=mode)
    ids = torch.as_tensor(image_ids).reshape(-1).to(image_emb.device)
    R = image_emb.shape[0]
    if ids.numel() != R:
        raise ValueError(f"image_ids has {ids.numel()} entries for {R} rows")
    uniq, inverse = torch.unique(ids, return_inverse=True)
    first = torch.full((uniq.numel(),), R, device=ids.device, dtype=torch.int64)
    first.scatter_reduce_(0, inverse, torch.arange(R, device=ids.device), reduce="amin")
    return retrieval_recall(text_emb, image_emb[first], inverse, ks=ks, mode=mode)
