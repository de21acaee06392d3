"""Retrieval top-k on the tensor cores (mc_retrieval_topk: threshold-and-collect epilogue of the resident pair kernel
plus a selection kernel per query) against an fp64 oracle.

The result is the exact top-k of the ENGINE's scores, so against fp64 it is held to a band: 3e-5 (tc_f16x3) and
2e-3 (tc_f16), absolute on cosines, as retrieval_ranks.  For every query: the indices are unique and in [0, N), the
values non-increasing, each value within the band of the fp64 score of its index; with v_k the k-th value,
#{fp64 > v_k + band} < k and #{fp64 >= v_k - band} >= k; and a query whose fp64 top-(k+1) has no gap narrower than
2 band returns exactly the fp64 top-k list, in order."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import retrieval_eval_ref as R

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _retrieval_pairs import make_pairs  # noqa: E402

pytestmark = pytest.mark.gpu
BAND = {"tc_f16x3": 3e-5, "tc_f16": 2e-3}


def _fp64_scores(text, image, rows):
    tn = F.normalize(text[rows].double(), p=2, dim=-1)
    xn = F.normalize(image.double(), p=2, dim=-1)
    return tn @ xn.T


def check_topk(text, image, k, vals, idx, mode, rows=None):
    """The fp64 checks of the module docstring for the queries `rows` (all by default), in blocks on the GPU.
    Returns the number of queries held to the exact fp64 list."""
    Q, N = text.shape[0], image.shape[0]
    band = BAND[mode]
    assert vals.shape == (Q, k) and idx.shape == (Q, k)
    assert vals.dtype == torch.float32 and idx.dtype == torch.int64
    rows = torch.arange(Q, device=text.device) if rows is None else rows.to(text.device)
    step = max(1, (1 << 24) // N)
    exact = 0
    for r0 in range(0, rows.numel(), step):
        rr = rows[r0:r0 + step]
        v, i = vals[rr].double(), idx[rr]
        assert ((i >= 0) & (i < N)).all()
        si = i.sort(1).values
        assert (si[:, 1:] != si[:, :-1]).all(), "repeated index"
        assert (v[:, 1:] <= v[:, :-1]).all(), "values not descending"
        S = _fp64_scores(text, image, rr)
        err = (v - S.gather(1, i)).abs()
        assert (err <= band).all(), float(err.max())
        vk = v[:, -1:]
        assert ((S > vk + band).sum(1) < k).all()
        assert ((S >= vk - band).sum(1) >= k).all()
        kk = min(k + 1, N)
        tv, ti = S.topk(kk, dim=1)
        gap = (tv[:, :-1] - tv[:, 1:]).min(1).values if kk > 1 else torch.full((rr.numel(),), float("inf"),
                                                                                 device=S.device, dtype=S.dtype)
        clear = gap >= 2 * band
        assert torch.equal(i[clear], ti[clear, :k])
        exact += int(clear.sum())
    return exact


def _topk(text, image, k, mode):
    import mae_clip_b200 as m
    return m.retrieval_topk(text, image, k, mode=mode)


def _randn(rows, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(rows, D, generator=g).cuda()


@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
@pytest.mark.parametrize("Q,N,D,k", [
    (1, 4097, 256, 10),        # one query: the bank is the resident side
    (127, 4097, 64, 100),      # Q << N
    (4097, 127, 128, 10),      # Q >> N: the queries are the resident side
    (129, 129, 100, 129),      # k == N, D not a multiple of 64
    (4097, 4097, 256, 1024),
    (1, 1, 64, 1),
    (127, 1, 128, 1),
    (4097, 129, 64, 100),
    (129, 127, 256, 1),
])
def test_shapes_against_fp64(Q, N, D, k, mode):
    text, image = _randn(Q, D, Q * 7 + D), _randn(N, D, N * 11 + D + 1)
    vals, idx = _topk(text, image, k, mode)
    exact = check_topk(text, image, k, vals, idx, mode)
    if mode == "tc_f16x3" and k <= 10 and Q > 1:
        assert exact >= 0.2 * Q   # the exact-list check is not vacuous


@pytest.mark.parametrize("Q,N,D,k", [
    (4097, 20000, 128, 100),   # bank rows: chunks of 7 936 rows, the last one ragged
    (40000, 5000, 64, 10),     # query rows: chunks of 768 columns, the last one ragged
])
def test_several_chunks(Q, N, D, k):
    text, image = _randn(Q, D, 5), _randn(N, D, 6)
    vals, idx = _topk(text, image, k, "tc_f16x3")
    rows = torch.randperm(Q, generator=torch.Generator().manual_seed(7))[:512]
    check_topk(text, image, k, vals, idx, "tc_f16x3", rows)


def _monotone_bank(Q, N, D, rising, seed):
    """Queries close to one direction u; bank row n = a_n u + noise with a_n monotone in n, so that every query's
    scores rise (or fall) along the bank: with rising scores each chunk replaces the whole running top-k and every
    candidate of every chunk after the first survives."""
    g = torch.Generator().manual_seed(seed)
    u = F.normalize(torch.randn(D, generator=g), dim=0)
    text = u + 0.01 * torch.randn(Q, D, generator=g)
    a = torch.linspace(-0.9, 0.9, N)
    if not rising:
        a = a.flip(0)
    image = a[:, None] * u + torch.sqrt(1 - a[:, None] ** 2) * F.normalize(torch.randn(N, D, generator=g), dim=1)
    return text.cuda(), image.cuda()


@pytest.mark.parametrize("rising", [True, False])
@pytest.mark.parametrize("Q,N,k", [(64, 200000, 100), (40000, 5000, 10)])
def test_monotone_banks(Q, N, k, rising):
    text, image = _monotone_bank(Q, N, 128, rising, seed=Q + N)
    vals, idx = _topk(text, image, k, "tc_f16x3")
    rows = torch.randperm(Q, generator=torch.Generator().manual_seed(3))[:256]
    check_topk(text, image, k, vals, idx, "tc_f16x3", rows)
    # the winners come from the last (rising) or first (falling) tenth of the bank
    assert ((idx >= N - N // 10) if rising else (idx < N // 10)).all()


def _assert_ties_to_lower_index(vals, idx, group):
    """Equal values come in ascending index order, and an index is returned only together with every lower index of
    the same duplicate group (the same bank row scores bit-identically)."""
    v, i = vals.cpu(), idx.cpu()
    same = v[:, 1:] == v[:, :-1]
    assert (i[:, 1:][same] > i[:, :-1][same]).all()
    g = group.cpu()
    for q in range(i.shape[0]):
        got = set(i[q].tolist())
        for n in got:
            lower = (g[:n] == g[n]).nonzero().flatten().tolist()
            assert set(lower) <= got, (q, n, lower[:5])


@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
def test_duplicated_bank_rows(mode):
    g = torch.Generator().manual_seed(41)
    base = torch.randn(300, 96, generator=g)
    group = torch.randint(0, 300, (5000,), generator=g)
    image = base[group].cuda()
    text = torch.randn(200, 96, generator=g).cuda()
    vals, idx = _topk(text, image, 50, mode)
    check_topk(text, image, 50, vals, idx, mode)
    assert (vals[:, 1:] == vals[:, :-1]).any(1).float().mean() > 0.5   # ties do occur in the lists
    _assert_ties_to_lower_index(vals, idx, group)


@pytest.mark.parametrize("Q,N", [(3, 70000), (3000, 300)])
def test_all_identical_bank(Q, N):
    text = _randn(Q, 128, 1)
    image = _randn(1, 128, 2).expand(N, 128).contiguous()
    vals, idx = _topk(text, image, 100, "tc_f16x3")
    assert torch.equal(idx.cpu(), torch.arange(100).expand(Q, 100))
    assert (vals == vals[:, :1]).all()


def test_zero_norm_rows_score_zero():
    text, image = _randn(300, 64, 3), _randn(3000, 64, 4)
    text[::7] = 0
    image[::5] = 0
    vals, idx = _topk(text, image, 700, "tc_f16x3")
    check_topk(text, image, 700, vals, idx, "tc_f16x3")
    zero_q = torch.arange(0, 300, 7)
    assert torch.equal(idx[zero_q].cpu(), torch.arange(700).expand(len(zero_q), 700))
    assert (vals[zero_q] == 0).all()
    # a zero bank row scores exactly 0 for every query
    z = idx % 5 == 0
    assert (vals[z] == 0).all()


@pytest.mark.parametrize("mode", ["tc_f16x3", "tc_f16"])
@pytest.mark.parametrize("n,D", [(1000, 256), (2000, 64)])
def test_consistent_with_retrieval_ranks(n, D, mode):
    """One-to-one pairs: caption q's own image is in its top-k exactly when its text->image rank is below k, and the
    same with the roles swapped (the image's captions against image->text ranks).

    Both rank the candidates by the same engine scores, but retrieval_ranks takes the positive's own score, the
    threshold, in fp32 (one warp per caption).  With tc_f16x3 the two thresholds agree to ~1e-7 and the membership
    must match exactly.  With tc_f16 (one fp16 pass) the engine's positive score differs from the fp32 one by up to
    the band, so a query may differ only when a candidate's fp64 score lies within twice the band of its positive's."""
    import mae_clip_b200 as m
    text, image = make_pairs(n, n, D, seed=n + D + 1)
    text, image = text.cuda(), image.cuda()
    t2i, i2t = m.retrieval_ranks(text, image, mode=mode)
    _, _, near_t, near_i = R.ranks_ref(text, image, band=2 * BAND[mode])
    own = torch.arange(n, device="cuda")[:, None]
    for k in (1, 5, 10):
        for rank, near, (a, b) in ((t2i, near_t, (text, image)), (i2t, near_i, (image, text))):
            _, idx = m.retrieval_topk(a, b, k, mode=mode)
            differ = (rank < k) != (idx == own).any(1)
            if mode == "tc_f16x3":
                assert not differ.any(), (k, differ.nonzero().flatten()[:5].tolist())
            else:
                assert (near[differ] > 0).all() and differ.double().mean() < 0.05, (k, int(differ.sum()))


def test_deterministic():
    for text, image, k in ((_randn(1000, 256, 8), _randn(50000, 256, 9), 100),
                           (*_monotone_bank(64, 200000, 128, True, seed=5), 1000)):   # heavy survivor traffic
        v1, i1 = _topk(text, image, k, "tc_f16x3")
        v2, i2 = _topk(text, image, k, "tc_f16x3")
        assert torch.equal(i1, i2)
        assert torch.equal(v1.view(torch.int32), v2.view(torch.int32))


def test_empty_queries():
    vals, idx = _topk(_randn(0, 64, 1)[:0], _randn(10, 64, 2), 5, "tc_f16x3")
    assert vals.shape == (0, 5) and idx.shape == (0, 5)


def test_errors():
    import mae_clip_b200 as m
    from mae_clip_b200._lib import MaeClipB200Error
    t, x = _randn(4, 64, 1), _randn(2000, 64, 2)
    with pytest.raises(ValueError, match="D <= 256"):
        m.retrieval_topk(_randn(4, 320, 1), _randn(10, 320, 2), 3)
    with pytest.raises(ValueError, match="D % 4"):
        m.retrieval_topk(_randn(4, 6, 1), _randn(10, 6, 2), 3)
    with pytest.raises(RuntimeError, match="out of range"):
        m.retrieval_topk(t, x[:10], 11)
    with pytest.raises(ValueError, match="k <= 1024"):
        m.retrieval_topk(t, x, 1025)
    with pytest.raises(MaeClipB200Error, match="tensor cores only"):
        m.retrieval_topk(t, x, 3, mode="simt_fp32")
    with pytest.raises(MaeClipB200Error):
        m.retrieval_topk(t.cpu(), x.cpu(), 3)
    with pytest.raises(ValueError, match="same D"):
        m.retrieval_topk(t, _randn(10, 128, 2), 3)
    with pytest.raises((ValueError, MaeClipB200Error)):
        m.retrieval_topk(t, x.cpu(), 3)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="same device"):
            m.retrieval_topk(t, x.to("cuda:1"), 3)


def test_at_scale_1024_queries_1m_bank():
    """Q = 1024 against N = 1 048 576, D = 256: a seeded sample of queries against the fp64 oracle, and the
    workspace stays below the documented formula and far below the Q x N score matrix."""
    import mae_clip_b200 as m
    from mae_clip_b200._lib import lib
    Q, N, D = 1024, 1 << 20, 256
    text, image = _randn(Q, D, 11), _randn(N, D, 12)
    rows = torch.randperm(Q, generator=torch.Generator().manual_seed(13))[:48]
    for k, mode in ((100, "tc_f16x3"), (10, "tc_f16")):
        vals, idx = m.retrieval_topk(text, image, k, mode=mode)
        check_topk(text, image, k, vals, idx, mode, rows)
        ws = lib().mc_retrieval_topk_workspace_bytes(Q, N, D, k, 1)
        C = 32768   # 2^28 / (8 Q)
        formula = 4 * Q * D + 4 * N * D + 4 * Q * D + 8 * Q * k + 8 * Q + 8 * Q * C + 16 * 256
        assert ws <= formula and ws < Q * N * 4 / 3


def test_ranks_unchanged_by_shared_prologue():
    """retrieval_ranks still matches its fp64 oracle after the prologue moved into the helper both entry points share."""
    import mae_clip_b200 as m
    text, image = make_pairs(3000, 1000, 128, seed=77, text_to_image=torch.arange(3000) % 1000)
    tti = (torch.arange(3000) % 1000).cuda()
    t2i, i2t = m.retrieval_ranks(text.cuda(), image.cuda(), tti)
    rt, ri, bt, bi = R.ranks_ref(text.cuda(), image.cuda(), tti, band=BAND["tc_f16x3"])
    assert ((t2i - rt).abs() <= bt).all() and ((i2t - ri).abs() <= bi).all()
