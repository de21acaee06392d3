"""Host-side checks of the retrieval top-k (no GPU): the workspace follows the formula of the header and has no
queries x bank term; CPU tensors are refused."""
import pytest
import torch


def _formula(Q, N, D, k):
    unit = 128 if Q >= N else 256
    C = max((2 ** 28 // (8 * Q)) // unit * unit, unit)
    C = min(C, 65536, -(-N // unit) * unit)
    Dp = -(-D // 8) * 8
    return 4 * Q * D + 4 * N * D + 4 * min(Q, N) * Dp + 8 * Q * k + 8 * Q + 8 * Q * C, C


@pytest.mark.parametrize("Q,N,D,k", [(1, 1 << 20, 256, 10), (1024, 1 << 20, 256, 100), (25000, 5000, 256, 10),
                                     (5000, 25000, 256, 10), (4097, 20000, 128, 100), (1, 1, 4, 1)])
def test_workspace_formula(lib_built, Q, N, D, k):
    from mae_clip_b200._lib import lib
    ws = lib().mc_retrieval_topk_workspace_bytes(Q, N, D, k, 1)
    f, C = _formula(Q, N, D, k)
    assert f <= ws <= f + 16 * 256
    # no Q x N term: a bank 16 times larger adds its own rows only
    ws16 = lib().mc_retrieval_topk_workspace_bytes(Q, 16 * N, D, k, 1)
    f16, C16 = _formula(Q, 16 * N, D, k)
    assert ws16 - ws <= 4 * 15 * N * D + 4 * min(Q, 16 * N) * D + 8 * Q * (C16 - C) + 16 * 256


def test_workspace_zero_for_empty_problems(lib_built):
    from mae_clip_b200._lib import lib
    assert lib().mc_retrieval_topk_workspace_bytes(0, 10, 64, 1, 1) == 0
    assert lib().mc_retrieval_topk_workspace_bytes(4, 10, 64, 0, 1) == 0


def test_cpu_tensors_refused():
    import mae_clip_b200 as m
    from mae_clip_b200._lib import MaeClipB200Error
    with pytest.raises(MaeClipB200Error, match="no CPU fallback"):
        m.retrieval_topk(torch.randn(4, 64), torch.randn(10, 64), 3)
