"""Retrieval evaluation without a device: the oracle on a hand-built example with known ranks, and the product path
refusing CPU tensors."""
import pytest
import torch

from oracle import retrieval_eval_ref as R


def _example():
    # 3 captions, 3 images; captions 0 and 1 describe image 0, caption 2 image 1; image 2 has no caption
    image = torch.tensor([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 1.0, 0]])
    text = torch.tensor([[1.0, 0.5, 0, 0], [0.2, 1.0, 0, 0], [0, 0.3, 1.0, 0]])
    return text, image, torch.tensor([0, 0, 1])


def test_ranks_ref_hand_built():
    text, image, tti = _example()
    t2i, i2t = R.ranks_ref(text, image, tti)
    # caption 0: own image first; caption 1: image 1 beats image 0; caption 2: image 2 beats image 1
    assert t2i.tolist() == [0, 1, 1]
    # image 0: best caption (0) first; image 1: captions 0 and 1 beat its caption 2; image 2: no caption
    assert i2t.tolist() == [0, 2, -1]
    _, _, bt, bi = R.ranks_ref(text, image, tti, band=1e-6)
    assert bt.tolist() == [0, 0, 0] and bi.tolist() == [0, 0, 0]


def test_recall_ref_hand_built():
    text, image, tti = _example()
    r = R.recall_ref(text, image, tti, ks=(1, 2, 3))
    assert r["text_to_image_R@1"] == pytest.approx(1 / 3) and r["text_to_image_R@2"] == 1.0
    # the image without a caption is left out: 1 of 2 at K = 1, 2 of 2 at K = 3
    assert r["image_to_text_R@1"] == 0.5 and r["image_to_text_R@2"] == 0.5 and r["image_to_text_R@3"] == 1.0


def test_ranks_ref_one_to_one_ties_favour_the_positive():
    image = torch.tensor([[1.0, 0], [1.0, 0], [0, 1.0]])
    text = torch.tensor([[2.0, 0], [1.0, 0], [1.0, 1.0]])
    t2i, i2t = R.ranks_ref(text, image)
    # captions 0 and 1 tie with the other identical image: a tie does not count
    assert t2i.tolist() == [0, 0, 0] and i2t.tolist() == [0, 0, 0]


def test_cpu_tensors_raise():
    import mae_clip_b200 as m
    from mae_clip_b200._lib import MaeClipB200Error
    text, image, tti = _example()
    with pytest.raises(MaeClipB200Error):
        m.retrieval_ranks(text, image, tti)
    with pytest.raises(MaeClipB200Error):
        m.retrieval_recall(text, image, tti)
