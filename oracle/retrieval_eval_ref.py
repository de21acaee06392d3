"""Oracle for the retrieval evaluation (``mae_clip_b200.retrieval_ranks`` / ``retrieval_recall``).

TEST INFRASTRUCTURE - see ``oracle/__init__.py``.  Not in the reference: the standard evaluation of a CLIP model,
recall@K in both directions (COCO / Karpathy-split convention for image->text: the rank of the best-ranked caption).

Restated with plain torch ops - ``F.normalize`` on both sides as ``inference.py:42-43``, matmul, comparisons -
chunked over queries so that the (Q, N) matrix is never whole.  Runs on the device of its inputs, in fp64 by default.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _normalized(text, image, text_to_image, dtype):
    tn = F.normalize(text.to(dtype), p=2, dim=-1)
    xn = F.normalize(image.to(dtype), p=2, dim=-1)
    Q = tn.shape[0]
    g = (torch.arange(Q, device=tn.device) if text_to_image is None
         else torch.as_tensor(text_to_image).to(device=tn.device, dtype=torch.int64))
    return tn, xn, g


def _chunks(Q, N, chunk):
    step = chunk or max(1, (1 << 24) // max(N, 1))
    for q0 in range(0, Q, step):
        yield q0, min(Q, q0 + step)


def _thresholds(tn, xn, g, chunk):
    """t[q] = s[q, g(q)]; u[n] = max over the captions of image n (-inf without one); has[n]."""
    Q, N = tn.shape[0], xn.shape[0]
    t = torch.empty(Q, dtype=tn.dtype, device=tn.device)
    for q0, q1 in _chunks(Q, N, chunk):
        s = tn[q0:q1] @ xn.T
        t[q0:q1] = s[torch.arange(q1 - q0, device=s.device), g[q0:q1]]
    u = torch.full((N,), float("-inf"), dtype=tn.dtype, device=tn.device)
    u.scatter_reduce_(0, g, t, reduce="amax")
    has = torch.zeros(N, dtype=torch.bool, device=tn.device)
    has[g] = True
    return t, u, has


def ranks_ref(text, image, text_to_image=None, dtype=torch.float64, chunk=None, band=None):
    """(t2i_rank (Q,), i2t_rank (N,)) int64, as mae_clip_b200.retrieval_ranks defines them: the number of
    non-positive candidates scoring strictly above the positive's score (the best positive's for an image); -1 for an
    image without a caption.  ``band``: also return, per caption and per image, the number of non-positive candidates
    whose score lies within ``band`` of the threshold (the candidates an engine of that accuracy may count either way)."""
    tn, xn, g = _normalized(text, image, text_to_image, dtype)
    Q, N = tn.shape[0], xn.shape[0]
    t, u, has = _thresholds(tn, xn, g, chunk)
    t2i = torch.zeros(Q, dtype=torch.int64, device=tn.device)
    i2t = torch.zeros(N, dtype=torch.int64, device=tn.device)
    bt = torch.zeros(Q, dtype=torch.int64, device=tn.device)
    bi = torch.zeros(N, dtype=torch.int64, device=tn.device)
    cols = torch.arange(N, device=tn.device)
    for q0, q1 in _chunks(Q, N, chunk):
        s = tn[q0:q1] @ xn.T
        neg = g[q0:q1, None] != cols[None, :]
        t2i[q0:q1] = ((s > t[q0:q1, None]) & neg).sum(1)
        i2t += ((s > u[None, :]) & neg).sum(0)
        if band is not None:
            bt[q0:q1] = (((s - t[q0:q1, None]).abs() <= band) & neg).sum(1)
            bi += (((s - u[None, :]).abs() <= band) & neg).sum(0)
    i2t[~has] = -1
    bi[~has] = 0
    return (t2i, i2t, bt, bi) if band is not None else (t2i, i2t)


def recall_from_ranks(t2i, i2t, ks=(1, 5, 10)):
    out = {}
    for k in ks:
        out[f"text_to_image_R@{k}"] = ((t2i >= 0) & (t2i < k)).double().mean().item()
    has = i2t >= 0
    for k in ks:
        out[f"image_to_text_R@{k}"] = (((i2t >= 0) & (i2t < k)).double().sum() / has.sum()).item() if has.any() \
            else float("nan")
    return out


def recall_ref(text, image, text_to_image=None, ks=(1, 5, 10), dtype=torch.float64, chunk=None):
    """{"text_to_image_R@K": ..., "image_to_text_R@K": ...}: fraction of captions / images with 0 <= rank < K (images
    without a caption are left out)."""
    return recall_from_ranks(*ranks_ref(text, image, text_to_image, dtype, chunk), ks)
