"""Golden fixtures for the MAE rows (M1-M3) from a PUBLISHED implementation.

``/root/reference`` holds no MAE code (SURVEY.md section 0.2), so the MAE oracle cannot be pinned on the
reference itself.  The formulation BASELINE.json names (noise argsort, keep / restore gather, normalised-pixel
masked-patch MSE) is the one of "Masked Autoencoders Are Scalable Vision Learners"; its implementation in
``transformers`` (``ViTMAEEmbeddings.random_masking``, ``ViTMAEForPreTraining.patchify / forward_loss``;
version recorded in the fixture) is importable here, so its outputs pin ``oracle/mae_ref.py`` and the CUDA path:

    python tests/golden/make_golden_mae.py        # writes tests/golden/mae_hf.npz

Every ``ref_`` array is an output of the transformers code run unmodified on CPU, and so is every ``mask`` of the MSE
cases; the seeded inputs are drawn by ``tests/_golden_inputs.py`` and stored only as digests (``<key>.sha256``).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
import transformers
from transformers import ViTMAEConfig, ViTMAEForPreTraining

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _golden_inputs as gi  # noqa: E402


def tiny_model(image_size, mask_ratio, norm_pix):
    cfg = ViTMAEConfig(hidden_size=32, num_hidden_layers=1, num_attention_heads=2, intermediate_size=64,
                       decoder_hidden_size=32, decoder_num_hidden_layers=1, decoder_num_attention_heads=2,
                       decoder_intermediate_size=64, image_size=image_size, patch_size=16, num_channels=3,
                       mask_ratio=mask_ratio, norm_pix_loss=norm_pix)
    return ViTMAEForPreTraining(cfg).eval()


def main():
    inputs = gi.mae_hf_inputs()
    out = {"transformers_version": np.array(transformers.__version__), **gi.digests(inputs)}
    # ---- M1: random masking at the reference patch count (196) and a ragged one, ratios of config C5
    for tag in gi.MASK_SHAPES:
        x, noise = torch.from_numpy(inputs[f"mask.{tag}.x"]), torch.from_numpy(inputs[f"mask.{tag}.noise"])
        for ratio in (0.5, 0.6, 0.75, 0.9):
            m = tiny_model(224, ratio, True)
            with torch.no_grad():
                xm, mask, ids_restore = m.vit.embeddings.random_masking(x, noise)
            k = f"mask.{tag}.r{int(ratio * 100)}"
            out[k + ".ref_x_masked"], out[k + ".ref_mask"], out[k + ".ref_ids_restore"] = \
                xm.numpy(), mask.numpy(), ids_restore.numpy()
    # ---- M2 + M3: patchify, normalised-pixel target (through the loss), masked MSE and its gradient
    for tag, (N, size) in gi.MSE_SHAPES.items():
        L = (size // 16) ** 2
        imgs, pred, noise = (torch.from_numpy(inputs[f"mse.{tag}.{k}"]) for k in ("imgs", "pred", "noise"))
        for norm_pix in ((True, False) if size == 64 else (True,)):  # keep the fixture small: 224 px once
            m = tiny_model(size, 0.75, norm_pix)
            with torch.no_grad():
                _, mask, _ = m.vit.embeddings.random_masking(torch.zeros(N, L, 4), noise)
                patches = m.patchify(imgs)
            p = pred.clone().requires_grad_(True)
            loss = m.forward_loss(imgs, p, mask)
            loss.backward()
            k = f"mse.{tag}.np{int(norm_pix)}"
            out[k + ".mask"] = mask.numpy()
            out[k + ".ref_loss"] = loss.detach().numpy()
            out[k + ".ref_dpred"] = p.grad.numpy()
            if norm_pix and size == 64:
                out[f"mse.{tag}.ref_patchify"] = patches.numpy()
    np.savez_compressed(os.path.join(HERE, "mae_hf.npz"), **out)
    print("wrote mae_hf.npz with", len(out), "arrays")


if __name__ == "__main__":
    main()
