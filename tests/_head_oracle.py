"""ProjectionHead runs against the fp64 oracle on the GPU, with per-block error metrics (tests/test_gpu_head_edges.py).

`proj_head_fwd_bwd_ref` is plain torch: in float64 on the GPU it keeps B = 32768, E = 2048 to a fraction of a second.
Inputs are row slices `buf[:B]` of larger buffers whose rows past B hold 1e4-scale values, so that a kernel reading a
row past B shows up as a large error instead of landing on zeros."""
import torch

from conftest import rel_err
from oracle import proj_head_ref

GRAD_NAMES = ["w_proj", "b_proj", "w_fc", "b_fc", "ln_w", "ln_b"]
POISON = 1e4
TAIL = 160          # rows of poison past B: more than a 128-row block


def expected_path(mode, B, E, P=256):
    """The path mc_proj_head_fwd / _bwd take (csrc/proj_head.cu: use_tc needs a tensor-core mode and B >= kTcMinRows
    = 2048; use_pair also needs hg::supported(P), i.e. P == 256, and E % 4 == 0 - its tile bound (E + 255) / 256 <=
    SMs / 2 holds for every E here)."""
    tc = mode in ("tc_f16x3", "tc_f16") and B >= 2048
    if tc and P == 256 and E % 4 == 0:
        return "pair"
    return "tc" if tc else "simt"


def path_of_launches(n):
    """Which path a forward took, from its kernel launch count (mc_kernel_launch_count): the FMA path launches two
    sgemm_kernel and one ln_fwd_kernel; the pair path a max|x| reduction (or, with a previous call's scale, the gated
    redo of the first GEMM), stage_pair_kernel and two row_kernel; the round-1 tensor-core path stages four operands
    (two launches each) around its two GEMMs and ln_fwd_kernel."""
    return {3: "simt", 4: "pair"}.get(n, "tc" if n > 4 else "?")


def make_head(E, mode, P=256, seed=0, p_drop=0.1):
    import mae_clip_b200 as m
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    h = m.ProjectionHead(E, projection_dim=P, gemm_mode=mode)
    h.dropout.p = p_drop
    with torch.no_grad():   # LayerNorm affine away from (1, 0), as tests/test_gpu_heads_model.py does
        h.layer_norm.weight.mul_(0.5).add_(torch.randn(P, generator=g) * 0.05)
        h.layer_norm.bias.add_(torch.randn(P, generator=g) * 0.1)
    return h.cuda().train()


def poisoned(shape, B, fill, gen, dtype=torch.float32):
    """`fill(buf)` fills a (B + TAIL, ...) buffer; rows past B are then set to POISON.  Returns the view buf[:B]."""
    buf = torch.empty((B + TAIL,) + tuple(shape[1:]), device="cuda", dtype=dtype)
    fill(buf, gen)
    buf[B:] = POISON if dtype.is_floating_point else 1
    return buf[:B]


def make_inputs(B, E, P=256, seed=0, p_drop=0.1, x_scale=1.0, special_rows=False):
    """x (B, E), keep (B, P) uint8 with P(keep) = 1 - p_drop, grad_out (B, P): row slices of poisoned buffers.
    `special_rows`: rows 0, 5 and B - 1 of keep all zero, rows 1 and B - 2 all one."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = poisoned((B, E), B, lambda b, g: b.normal_(generator=g).mul_(x_scale), gen)
    keep = poisoned((B, P), B, lambda b, g: b.copy_(torch.rand(b.shape, device="cuda", generator=g) >= p_drop), gen,
                    torch.uint8)
    if special_rows:
        keep[[0, 5, B - 1]] = 0
        keep[[1, B - 2]] = 1
    go = poisoned((B, P), B, lambda b, g: b.normal_(generator=g), gen)
    return x, keep, go


def run_head(h, x, keep, go, need_dx):
    """Forward (train mode with `keep`, or eval mode when h is in eval) and backward through autograd.  Returns
    (out, grads, path) with grads keyed as the oracle's and path read from the forward's launch count."""
    from mae_clip_b200 import _lib
    xc = x.requires_grad_(need_dx)
    n0 = _lib.lib().mc_kernel_launch_count()
    out = h(xc, keep_mask=keep if h.training else None)
    n1 = _lib.lib().mc_kernel_launch_count()
    out.backward(go)
    grads = {n: p.grad for n, p in zip(GRAD_NAMES, h.parameters())}
    grads["x"] = xc.grad
    if need_dx:
        xc.grad = None
    for p in h.parameters():
        p.grad = None
    return out.detach(), grads, path_of_launches(n1 - n0)


def oracle(h, x, keep, go, need_dx=True):
    """fp64 forward + backward of the head's current weights, on the GPU."""
    params = [p.detach() for p in h.parameters()]
    return proj_head_ref.proj_head_fwd_bwd_ref(x, params, keep if h.training else None, h.dropout.p, go,
                                               need_dx=need_dx, dtype=torch.float64)


def tile_errors(d, ref, rows=128, cols=None):
    """Relative error of every rows x cols tile, ||d_t - ref_t|| / ||ref_t|| on RMS values so that a ragged last tile
    weighs like a full one (as test_gpu_loss_edges.py's _block_errors).  A tile whose reference RMS is below a tenth
    of the median tile's is measured against that tenth.  Returns a (row tiles, column tiles) float64 tensor."""
    d, ref = d.double(), ref.double().to(d.device)
    R, C = ref.shape
    cols = cols or C
    nr, nc = -(-R // rows), -(-C // cols)
    pad = (0, nc * cols - C, 0, nr * rows - R)

    def norms(t):
        t = torch.nn.functional.pad(t, pad).reshape(nr, rows, nc, cols)
        return t.square().sum(dim=(1, 3)).sqrt()
    n_r = torch.full((nr, 1), float(rows), dtype=torch.float64, device=d.device)
    n_r[-1] = R - (nr - 1) * rows
    n_c = torch.full((1, nc), float(cols), dtype=torch.float64, device=d.device)
    n_c[0, -1] = C - (nc - 1) * cols
    n = (n_r * n_c).sqrt()
    rms = norms(ref) / n
    floor = (0.1 * rms.median()).clamp_min(torch.finfo(torch.float64).tiny)   # an all-zero reference (x = 0: dW_proj)
    return (norms(d - ref) / n / torch.maximum(rms, floor)).cpu()


def head_errors(out, grads, out_ref, grads_ref):
    """Whole-tensor relative errors of every output and gradient, and the per-block ones: out and dx per 128-row block
    (one CTA's rows; `*_last` = the possibly ragged last block), dW_proj and dW_fc per 128 x 256 tile."""
    e = {"out": rel_err(out, out_ref)}
    for n in GRAD_NAMES + ["x"]:
        if grads_ref[n] is not None:
            e[n] = rel_err(grads[n], grads_ref[n])
    for n, t, r, cols in (("out", out, out_ref, None), ("x", grads["x"], grads_ref["x"], None),
                          ("w_proj", grads["w_proj"], grads_ref["w_proj"], 256),
                          ("w_fc", grads["w_fc"], grads_ref["w_fc"], 256)):
        if r is None:
            continue
        b = tile_errors(t, r, 128, cols)
        e[n + "_block"] = b.max().item()
        if cols is None:
            e[n + "_last"] = b[-1].max().item()
    return e


def nonfinite(out, grads):
    """Names of the outputs / gradients holding a NaN or inf."""
    ts = {"out": out, **grads}
    return [n for n, t in ts.items() if t is not None and not bool(torch.isfinite(t).all())]
