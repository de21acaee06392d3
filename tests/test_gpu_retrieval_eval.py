"""Retrieval evaluation on the tensor cores (mc_retrieval_ranks: rank counts in the epilogue of the resident pair
kernel) against the fp64 oracle oracle/retrieval_eval_ref.py.

Band rule: the kernel compares the engine's scores, so a non-positive candidate whose true score lies within the
engine's rounding of the threshold may be counted on either side.  For every caption and image the returned rank may
differ from the fp64 rank by at most the number of such candidates (fp64 score within BAND[mode] of the fp64
threshold), and at least 90 % of them must have none, so that the comparison is not vacuous."""
import os
import sys

import pytest
import torch

from oracle import retrieval_eval_ref as R

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _retrieval_pairs import make_pairs  # noqa: E402

pytestmark = pytest.mark.gpu
BAND = {"tc_f16x3": 3e-5, "tc_f16": 2e-3}


def _check(text, image, tti, mode="tc_f16x3", recall_range=(0.2, 0.8)):
    import mae_clip_b200 as m
    tc, xc = text.cuda(), image.cuda()
    ttic = None if tti is None else tti.cuda()
    t2i, i2t = m.retrieval_ranks(tc, xc, ttic, mode=mode)
    assert t2i.dtype == torch.int64 and i2t.dtype == torch.int64
    assert t2i.shape == (text.shape[0],) and i2t.shape == (image.shape[0],)
    rt, ri, bt, bi = R.ranks_ref(tc, xc, ttic, band=BAND[mode])
    for got, ref, band, name in ((t2i, rt, bt, "text->image"), (i2t, ri, bi, "image->text")):
        has = ref >= 0
        assert torch.equal(got < 0, ref < 0), name              # -1 exactly for the images without a caption
        diff = (got - ref).abs()
        bad = diff > band
        assert not bad.any(), (name, int(bad.sum()), (got[bad][:5].tolist(), ref[bad][:5].tolist(), band[bad][:5].tolist()))
        assert (band[has] == 0).double().mean().item() >= 0.9, name
    if recall_range is not None:
        r1 = ((rt >= 0) & (rt < 1)).double().mean().item()
        assert recall_range[0] <= r1 <= recall_range[1], r1   # the counts are not trivial
    return t2i, i2t, rt, ri, bt, bi


@pytest.mark.parametrize("n", [1000, 4097])
@pytest.mark.parametrize("D", [256, 128, 64])
def test_one_to_one(n, D):
    text, image = make_pairs(n, n, D, seed=n + D)
    _check(text, image, None)


def test_coco_like_five_captions_per_image():
    g = torch.Generator().manual_seed(11)
    tti = torch.arange(1000).repeat_interleave(5)[torch.randperm(5000, generator=g)]
    text, image = make_pairs(5000, 1000, 256, seed=12, text_to_image=tti)
    _check(text, image, tti)


def test_ragged_mapping_with_uncaptioned_images():
    import mae_clip_b200 as m
    g = torch.Generator().manual_seed(21)
    tti = torch.randint(0, 3001, (777,), generator=g)
    text, image = make_pairs(777, 3001, 96, seed=22, text_to_image=tti)
    t2i, i2t, rt, ri, bt, bi = _check(text, image, tti)
    uncaptioned = torch.ones(3001, dtype=torch.bool)
    uncaptioned[tti] = False
    assert uncaptioned.sum() > 2000
    assert (i2t.cpu()[uncaptioned] == -1).all() and (i2t.cpu()[~uncaptioned] >= 0).all()
    r = m.retrieval_recall(text.cuda(), image.cuda(), tti.cuda(), ks=(1, 10))
    has = i2t >= 0
    assert r["image_to_text_R@10"] == pytest.approx(((i2t >= 0) & (i2t < 10)).sum().item() / has.sum().item(), abs=1e-12)


def test_row_blocks_split_across_pairs():
    """40 000 captions: 157 row blocks on at most 74 CTA pairs, so the remainder jobs split row blocks between pairs
    (row counts meet in atomics); 517 images is not a multiple of the 128-column tile."""
    g = torch.Generator().manual_seed(31)
    tti = torch.randint(0, 517, (40000,), generator=g)
    text, image = make_pairs(40000, 517, 256, seed=32, text_to_image=tti, k=0.8)
    _check(text, image, tti)


def test_images_on_the_resident_side():
    """300 captions x 70 000 images: the images are the larger set and take the resident (row) side."""
    g = torch.Generator().manual_seed(41)
    tti = torch.randperm(70000, generator=g)[:300]
    text, image = make_pairs(300, 70000, 256, seed=42, text_to_image=tti, k=1.0)
    _check(text, image, tti, recall_range=(0.2, 0.8))


def test_swapping_text_and_image_mirrors_the_ranks():
    import mae_clip_b200 as m
    text, image = make_pairs(4097, 4097, 256, seed=51)
    t2i, i2t, _, _, bt, bi = _check(text, image, None)
    t2i_s, i2t_s = m.retrieval_ranks(image.cuda(), text.cuda())
    # caption q against all images is image q against all captions of the swapped call; only the band may differ
    assert ((t2i - i2t_s).abs() <= bt).all() and ((i2t - t2i_s).abs() <= bi).all()
    assert (t2i == i2t_s).double().mean().item() > 0.97


def test_single_pass_engine_with_its_band():
    text, image = make_pairs(1000, 1000, 64, seed=61, k=1.0)
    _check(text, image, None, mode="tc_f16")


def test_zero_norm_rows_score_zero():
    text, image = make_pairs(1000, 1000, 128, seed=71)
    text[[3, 500, 999]] = 0
    image[[7, 500, 998]] = 0
    t2i, i2t, rt, ri, _, _ = _check(text, image, None)
    # a zero caption scores exactly 0 against everything: no image beats its own
    assert t2i[[3, 500, 999]].tolist() == [0, 0, 0] and rt[[3, 500, 999]].tolist() == [0, 0, 0]


def test_repeat_calls_are_identical():
    import mae_clip_b200 as m
    g = torch.Generator().manual_seed(81)
    tti = torch.randint(0, 2000, (9000,), generator=g)
    text, image = make_pairs(9000, 2000, 256, seed=82, text_to_image=tti)
    a = m.retrieval_ranks(text.cuda(), image.cuda(), tti.cuda())
    b = m.retrieval_ranks(text.cuda(), image.cuda(), tti.cuda())
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
def test_recall_matches_ranks_and_oracle(mode):
    import mae_clip_b200 as m
    g = torch.Generator().manual_seed(91)
    tti = torch.arange(1000).repeat_interleave(5)[torch.randperm(5000, generator=g)]
    text, image = make_pairs(5000, 1000, 256, seed=92, text_to_image=tti, k=1.0)
    tc, xc, ttic = text.cuda(), image.cuda(), tti.cuda()
    ks = (1, 5, 10)
    r = m.retrieval_recall(tc, xc, ttic, ks=ks, mode=mode)
    t2i, i2t = m.retrieval_ranks(tc, xc, ttic, mode=mode)
    ref = R.recall_ref(tc, xc, ttic, ks=ks)
    _, _, bt, bi = R.ranks_ref(tc, xc, ttic, band=BAND[mode])
    for k in ks:
        assert r[f"text_to_image_R@{k}"] == pytest.approx(((t2i >= 0) & (t2i < k)).double().mean().item(), abs=1e-12)
        assert r[f"image_to_text_R@{k}"] == pytest.approx(((i2t >= 0) & (i2t < k)).double().mean().item(), abs=1e-12)
        assert abs(r[f"text_to_image_R@{k}"] - ref[f"text_to_image_R@{k}"]) <= (bt > 0).sum().item() / 5000 + 1e-12
        assert abs(r[f"image_to_text_R@{k}"] - ref[f"image_to_text_R@{k}"]) <= (bi > 0).sum().item() / 1000 + 1e-12


def test_evaluate_retrieval_tiny_towers():
    import _tiny_towers as tt
    import mae_clip_b200 as m
    from mae_clip_b200.inference import _embed_pairs
    torch.manual_seed(0)
    model = m.CLIPModel(temperature=1.0, image_embedding=tt.IMG_DIM, text_embedding=tt.TXT_DIM,
                        image_encoder=tt.ImageTower(), text_encoder=tt.TextTower()).cuda()
    g = torch.Generator().manual_seed(101)
    n_img, rows, B, L = 40, 96, 24, 16
    images = torch.randn(n_img, 3, 32, 32, generator=g)
    image_ids = torch.cat([torch.arange(n_img), torch.randint(0, n_img, (rows - n_img,), generator=g)])
    image_ids = image_ids[torch.randperm(rows, generator=g)]
    ids = torch.randint(1, 400, (rows, L), generator=g)
    mask = torch.ones(rows, L, dtype=torch.long)
    loader = [{"image": images[image_ids[i:i + B]], "input_ids": ids[i:i + B], "attention_mask": mask[i:i + B]}
              for i in range(0, rows, B)]
    model.train()
    r = m.evaluate_retrieval(model, loader, ks=(1, 5, 10), image_ids=image_ids)
    assert model.training   # the caller's mode is restored
    img_emb, txt_emb = _embed_pairs(model, loader)
    uniq, inverse = torch.unique(image_ids, return_inverse=True)
    first = torch.tensor([int((image_ids == u).nonzero()[0]) for u in uniq])
    img_u, tti = img_emb[first.cuda()], inverse.cuda()
    ref = R.recall_ref(txt_emb, img_u, tti, ks=(1, 5, 10))
    _, _, bt, bi = R.ranks_ref(txt_emb, img_u, tti, band=BAND["tc_f16x3"])
    assert set(r) == set(ref)
    for k in (1, 5, 10):
        assert abs(r[f"text_to_image_R@{k}"] - ref[f"text_to_image_R@{k}"]) <= (bt > 0).sum().item() / rows + 1e-12
        assert abs(r[f"image_to_text_R@{k}"] - ref[f"image_to_text_R@{k}"]) <= (bi > 0).sum().item() / n_img + 1e-12
    # without image_ids: one-to-one rows
    r1 = m.evaluate_retrieval(model, loader, ks=(1,))
    ref1 = R.recall_ref(txt_emb, img_emb, None, ks=(1,))
    _, _, bt1, _ = R.ranks_ref(txt_emb, img_emb, None, band=BAND["tc_f16x3"])
    assert abs(r1["text_to_image_R@1"] - ref1["text_to_image_R@1"]) <= (bt1 > 0).sum().item() / rows + 1e-12


@pytest.mark.parametrize("D", [320, 6])
def test_unsupported_width_raises(D):
    import mae_clip_b200 as m
    from mae_clip_b200._lib import MaeClipB200Error
    x = torch.randn(64, D, device="cuda")
    with pytest.raises(MaeClipB200Error):
        m.retrieval_ranks(x, x)


def test_invalid_inputs_raise():
    import mae_clip_b200 as m
    from mae_clip_b200._lib import MaeClipB200Error
    t, x = torch.randn(10, 64, device="cuda"), torch.randn(8, 64, device="cuda")
    with pytest.raises(ValueError):
        m.retrieval_ranks(t, torch.randn(8, 32, device="cuda"), torch.zeros(10, dtype=torch.int64))
    with pytest.raises(ValueError):
        m.retrieval_ranks(t, x)   # Q != N needs a mapping
    bad = torch.arange(10, device="cuda")   # 8 and 9 are not images
    with pytest.raises(ValueError):
        m.retrieval_ranks(t, x, bad)
    with pytest.raises(ValueError):
        m.retrieval_recall(t, x, bad)
    with pytest.raises(ValueError):
        m.retrieval_recall(t, x, bad - 3)
    with pytest.raises(MaeClipB200Error):
        m.retrieval_ranks(t, x, bad % 8, mode="simt_fp32")
