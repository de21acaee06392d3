"""Seeded, correlated (caption, image) embedding pairs for the retrieval-evaluation tests (test infrastructure).

text = image[g(q)] + sigma * noise, both sides LayerNorm-ed as the projection heads produce them.  sigma follows the
largest negative score of random unit vectors, sqrt(2 ln N / D): the positive's expected cosine is k times that, so
that recall@1 lands between 0.2 and 0.8 for k around 0.8 - 0.9 (measured with the fp64 oracle)."""
import math

import torch
import torch.nn.functional as F


def sigma_for(n, D, k=0.9):
    c = k * math.sqrt(2 * math.log(n) / D)
    return math.sqrt(max(1 / c ** 2 - 1, 0.01))


def make_pairs(Q, N, D, seed, text_to_image=None, k=0.9):
    g = torch.Generator().manual_seed(seed)
    image = torch.randn(N, D, generator=g)
    gi = text_to_image if text_to_image is not None else torch.arange(N)
    text = image[gi] + sigma_for(max(Q, N), D, k) * torch.randn(Q, D, generator=g)
    return F.layer_norm(text, (D,)), F.layer_norm(image, (D,))
