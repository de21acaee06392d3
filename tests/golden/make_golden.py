"""Generate the golden fixtures by running the UNMODIFIED reference.

Run in the dev container only (needs ``/root/reference``):

    python tests/golden/make_golden.py

Writes ``tests/golden/*.npz``.  Every array under a ``ref_`` key is an output of
the reference's own code (its ``CLIP.py`` / ``modules.py``, imported through
``oracle/reference_shim.py``), and so are the dropout keep masks.  The seeded inputs
of ``clip_loss.npz`` and ``proj_head_model.npz`` are drawn by ``tests/_golden_inputs.py``
and stored only as digests (``<key>.sha256``).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _golden_inputs as gi  # noqa: E402
from oracle import reference_shim  # noqa: E402


class _TextStandIn(nn.Module):
    """Feeds pre-computed text features through the reference forward's keyword call
    (``CLIP.py:26-28``); the DistilBERT tower itself is out of scope (SURVEY section 2)."""

    def forward(self, input_ids, attention_mask):
        return input_ids


def _bare_clip_model(ref_clip, image_projection, text_projection, temperature):
    m = ref_clip.CLIPModel.__new__(ref_clip.CLIPModel)
    nn.Module.__init__(m)
    m.image_encoder = nn.Identity()
    m.text_encoder = _TextStandIn()
    m.image_projection = image_projection
    m.text_projection = text_projection
    m.temperature = temperature
    return m


def _np(t):
    return t.detach().cpu().numpy()


def gen_loss_cases(ref_clip):
    """Loss on given embeddings: reference ``CLIPModel.forward`` with identity heads, so
    lines ``CLIP.py:34-43`` run unmodified."""
    inputs = gi.clip_loss_inputs()
    out = gi.digests(inputs)
    for name, (_B, _scale, tau, _dup) in gi.LOSS_CASES.items():
        I, T = torch.from_numpy(inputs[f"{name}.I"]), torch.from_numpy(inputs[f"{name}.T"])
        for dt, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
            Ii = I.to(dt).clone().requires_grad_(True)
            Ti = T.to(dt).clone().requires_grad_(True)
            model = _bare_clip_model(ref_clip, nn.Identity(), nn.Identity(), tau)
            loss = model({"image": Ii, "input_ids": Ti, "attention_mask": None})
            loss.backward()
            out[f"{name}.ref_loss_{tag}"] = _np(loss)
            if tag == "f32":  # f64 gradients are covered by the closed-form oracle; keep fixtures small
                out[f"{name}.ref_dI_{tag}"] = _np(Ii.grad)
                out[f"{name}.ref_dT_{tag}"] = _np(Ti.grad)
        out[f"{name}.tau"] = np.float64(tau)
    np.savez_compressed(os.path.join(HERE, "clip_loss.npz"), **out)
    return len(gi.LOSS_CASES)


def gen_cross_entropy_cases(ref_clip):
    g = torch.Generator().manual_seed(3)
    out = {}
    preds = torch.randn(5, 7, generator=g) * 3
    targets = torch.softmax(torch.randn(5, 7, generator=g), dim=-1)
    sq_p = torch.randn(9, 9, generator=g) * 2
    sq_t = torch.softmax(torch.randn(9, 9, generator=g), dim=-1)
    out["rect.preds"], out["rect.targets"] = _np(preds), _np(targets)
    out["rect.ref_none"] = _np(ref_clip.cross_entropy(preds, targets, reduction="none"))
    out["rect.ref_mean"] = _np(ref_clip.cross_entropy(preds, targets, reduction="mean"))
    assert ref_clip.cross_entropy(preds, targets, reduction="sum") is None
    out["rect.ref_sum_is_none"] = np.array(True)
    out["sq.preds"], out["sq.targets"] = _np(sq_p), _np(sq_t)
    # the transposed-view call of CLIP.py:41 (targets.T rows do not sum to one)
    out["sq.ref_none_T"] = _np(ref_clip.cross_entropy(sq_p.T, sq_t.T, reduction="none"))
    p = sq_p.clone().requires_grad_(True)
    t = sq_t.clone().requires_grad_(True)
    w = torch.linspace(0.5, 1.5, 9)
    (ref_clip.cross_entropy(p.T, t.T, reduction="none") * w).sum().backward()
    out["sq.w"] = _np(w)
    out["sq.ref_dpreds_T"] = _np(p.grad)
    out["sq.ref_dtargets_T"] = _np(t.grad)
    np.savez_compressed(os.path.join(HERE, "cross_entropy.npz"), **out)


def gen_head_and_model_cases(ref_clip, ref_modules):
    """ProjectionHead alone (eval + train with the captured dropout mask) and the full
    heads+loss forward/backward of ``CLIPModel.forward``.  Small embedding dims keep the
    fixture small; ``embedding_dim`` is a constructor argument (``modules.py:58``)."""
    # the dropout masks below are drawn from the global generator where the seeded inputs leave it
    inputs = gi.proj_head_model_inputs()
    out = gi.digests(inputs)
    with torch.random.fork_rng(devices=[]):
        head_i = ref_modules.ProjectionHead(embedding_dim=gi.E_IMG)
        head_t = ref_modules.ProjectionHead(embedding_dim=gi.E_TXT)
    for tag, h in (("img", head_i), ("txt", head_t)):
        h.load_state_dict({k: torch.from_numpy(inputs[f"{tag}.{k}"]) for k in h.state_dict()})
    x_img, x_txt = torch.from_numpy(inputs["x_img"]), torch.from_numpy(inputs["x_txt"])

    # eval-mode head outputs
    head_i.eval(); head_t.eval()
    out["ref_eval_out_img"] = _np(head_i(x_img))
    out["ref_eval_out_txt"] = _np(head_t(x_txt))

    # train-mode: capture the dropout keep mask the reference drew
    masks = {}

    def hook(name):
        def fn(_m, inp, outp):
            masks[name] = (outp != 0) | (inp[0] == 0)
        return fn

    hi = head_i.dropout.register_forward_hook(hook("img"))
    ht = head_t.dropout.register_forward_hook(hook("txt"))
    head_i.train(); head_t.train()
    for tau, tag in ((1.0, "tau1"), (0.5, "tau05")):
        for p in list(head_i.parameters()) + list(head_t.parameters()):
            p.grad = None
        xi = x_img.clone().requires_grad_(True)
        xt = x_txt.clone().requires_grad_(True)
        model = _bare_clip_model(ref_clip, head_i, head_t, tau)
        model.train()
        loss = model({"image": xi, "input_ids": xt, "attention_mask": None})
        loss.backward()
        out[f"{tag}.keep_img"] = _np(masks["img"]).astype(np.uint8)
        out[f"{tag}.keep_txt"] = _np(masks["txt"]).astype(np.uint8)
        out[f"{tag}.ref_loss"] = _np(loss)
        out[f"{tag}.ref_dx_img"] = _np(xi.grad)
        out[f"{tag}.ref_dx_txt"] = _np(xt.grad)
        if tag == "tau1":  # parameter grads once; the second temperature pins loss + input grads
            for htag, h in (("img", head_i), ("txt", head_t)):
                for k, p in h.named_parameters():
                    out[f"{tag}.ref_grad.{htag}.{k}"] = _np(p.grad)
    hi.remove(); ht.remove()

    # eval-mode full forward (valid_epoch path, main.py:70-82)
    model = _bare_clip_model(ref_clip, head_i, head_t, 1.0)
    model.eval()
    with torch.no_grad():
        out["ref_eval_loss"] = _np(model({"image": x_img, "input_ids": x_txt, "attention_mask": None}))
    np.savez_compressed(os.path.join(HERE, "proj_head_model.npz"), **out)


def main():
    ref_clip, ref_modules = reference_shim.load()
    n = gen_loss_cases(ref_clip)
    gen_cross_entropy_cases(ref_clip)
    gen_head_and_model_cases(ref_clip, ref_modules)
    print(f"wrote fixtures ({n} loss cases) with torch {torch.__version__}")


if __name__ == "__main__":
    main()
