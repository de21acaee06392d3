"""Seeded inputs of the golden fixtures under ``tests/golden`` (test infrastructure).

A fixture stores what the reference computed.  The inputs it computed them from are drawn here from fixed seeds, by the
generator scripts and by the tests alike, instead of being stored a second time: that keeps every fixture under 1 MB.
Each fixture keeps the SHA-256 digest of every input it was made from (``<key>.sha256``) and ``regenerate`` checks them,
so a torch whose generators draw other numbers fails loudly instead of comparing the reference's outputs with results
for other inputs."""
import hashlib

import numpy as np
import torch
from torch import nn

from oracle.loss_ref import make_embeddings

# clip_loss.npz: case -> (rows, embedding scale, temperature, duplicated rows)
LOSS_CASES = {
    "b8_default": (8, 1.0, 1.0, False),
    "b48_soft_tau05": (48, 0.25, 0.5, False),
    "b33_dup_tau2": (33, 0.35, 2.0, True),
    "b130_soft": (130, 0.2, 1.0, False),
    # genuinely soft targets: Z_ii = 256 * 0.08^2 * tau / ... ~ 2, so P is far from one-hot and
    # the gradient through the (non-detached) targets is O(1) of the total
    "b64_verysoft": (64, 0.08, 1.5, True),
}

# proj_head_model.npz: embedding widths of the two heads and the batch; small widths keep the fixture small
# (``embedding_dim`` is a constructor argument, modules.py:58)
E_IMG, E_TXT, HEAD_BATCH = 160, 96, 24

# mae_hf.npz: random masking at the reference patch count (196) and a ragged one; masked MSE at 64 and 224 px
MASK_SHAPES = {"l196": (6, 196, 24), "l50": (4, 50, 8)}
MSE_SHAPES = {"s64": (3, 64), "s224": (1, 224)}


def clip_loss_inputs():
    out = {}
    for name, (B, scale, _tau, dup) in LOSS_CASES.items():
        I = make_embeddings(B, 256, seed=10, scale=scale)
        T = make_embeddings(B, 256, seed=11, scale=scale)
        if dup:
            I[5] = I[2]
            T[5] = T[2]
            T[7] = T[1]
        out[f"{name}.I"], out[f"{name}.T"] = I.numpy(), T.numpy()
    return out


def proj_head_model_inputs():
    """The initial state of the two reference heads and their input rows.  Seeds and draws from torch's global
    generator, in the reference's order: each ``ProjectionHead`` builds ``projection``, ``fc`` and ``layer_norm`` in
    that order (modules.py:55-67), then the LayerNorm affine is made non-trivial so its gradients are exercised."""
    torch.manual_seed(1234)
    heads = {}
    for tag, E in (("img", E_IMG), ("txt", E_TXT)):
        heads[tag] = {"projection": nn.Linear(E, 256), "fc": nn.Linear(256, 256), "layer_norm": nn.LayerNorm(256)}
    out = {}
    with torch.no_grad():
        for tag, h in heads.items():
            h["layer_norm"].weight.mul_(0.3).add_(torch.randn(256) * 0.02)
            h["layer_norm"].bias.add_(torch.randn(256) * 0.05)
            for layer, mod in h.items():
                out[f"{tag}.{layer}.weight"] = mod.weight.numpy().copy()
                out[f"{tag}.{layer}.bias"] = mod.bias.numpy().copy()
    out["x_img"] = torch.randn(HEAD_BATCH, E_IMG).numpy()
    out["x_txt"] = torch.randn(HEAD_BATCH, E_TXT).numpy()
    return out


def mae_hf_inputs():
    """``mse.*.noise`` only draws the mask the fixture stores (``mse.*.np*.mask``)."""
    g = torch.Generator().manual_seed(2024)
    out = {}
    for tag, (N, L, D) in MASK_SHAPES.items():
        out[f"mask.{tag}.x"] = torch.randn(N, L, D, generator=g).numpy()
        out[f"mask.{tag}.noise"] = torch.rand(N, L, generator=g).numpy()
    for tag, (N, size) in MSE_SHAPES.items():
        L = (size // 16) ** 2
        out[f"mse.{tag}.imgs"] = torch.randn(N, 3, size, size, generator=g).numpy()
        out[f"mse.{tag}.pred"] = (torch.randn(N, L, 768, generator=g) * 0.7).numpy()
        out[f"mse.{tag}.noise"] = torch.rand(N, L, generator=g).numpy()
    return out


SEEDED = {"clip_loss": clip_loss_inputs, "proj_head_model": proj_head_model_inputs, "mae_hf": mae_hf_inputs}


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def digests(inputs):
    """The ``<key>.sha256`` entries a generator stores next to the reference's outputs."""
    return {k + ".sha256": np.array(digest(v)) for k, v in inputs.items()}


def regenerate(name, stored):
    """The seeded inputs of fixture ``name``, checked against the digests ``stored`` in it."""
    with torch.random.fork_rng(devices=[]):
        inputs = SEEDED[name]()
    for k, v in inputs.items():
        if digest(v) != str(stored[k + ".sha256"]):
            raise AssertionError(f"{name}.npz: the seeded input {k} no longer reproduces (torch {torch.__version__} "
                                 "draws other numbers than the generator of the fixture did)")
    return inputs
