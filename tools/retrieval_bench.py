"""Retrieval evaluation timing: mae_clip_b200.retrieval_ranks (both tensor-core modes) against the eager torch
composition a user would otherwise write (F.normalize, fp32 matmul with TF32 off, comparisons; chunked over queries).

    python tools/retrieval_bench.py [--calls 20] [--out FILE.json] [--sizes flickr1k,coco5k,100k,300k]

Per size: median of per-call CUDA-event times over `--calls` calls after warm-up; the ranks kernel's own time from a
separate torch.profiler run; the executed tensor rate (passes x 2QND over kernel time) and the algorithmic rate (2QND
over call time); at the two smaller sizes a parity check of both modes' ranks against the fp64 oracle with the band
rule of tests/test_gpu_retrieval_eval.py.  D = 256.  Inputs: seeded correlated pairs, text = image + noise, LayerNorm-ed.
The card's name, power limit and maximum SM clock are read with nvidia-smi (a query only) and stored with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

SIZES = {  # name: (Q captions, N images, captions per image)
    "flickr1k": (5000, 1000, 5),
    "coco5k": (25000, 5000, 5),
    "100k": (100000, 100000, 1),
    "300k": (300000, 300000, 1),
}
BAND = {"tc_f16x3": 3e-5, "tc_f16": 2e-3}
PASSES = {"tc_f16x3": 3, "tc_f16": 1}
D = 256


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"nvidia_smi": out}


def make_inputs(Q, N, per, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    image = torch.randn(N, D, device="cuda", generator=g)
    if per == 1:
        tti = None
        gi = torch.arange(N, device="cuda")
    else:
        gi = torch.arange(N, device="cuda").repeat_interleave(per)
        gi = gi[torch.randperm(Q, device="cuda", generator=g)]
        tti = gi
    text = image[gi] + 4.0 * torch.randn(Q, D, device="cuda", generator=g)
    return F.layer_norm(text, (D,)), F.layer_norm(image, (D,)), tti


def torch_ranks(text, image, tti, chunk_bytes=4 << 30):
    """The eager composition: fp32, TF32 off (the reference's precision), chunked over queries."""
    Q, N = text.shape[0], image.shape[0]
    tn, xn = F.normalize(text, p=2, dim=-1), F.normalize(image, p=2, dim=-1)
    g = tti if tti is not None else torch.arange(Q, device=text.device)
    t = (tn * xn[g]).sum(-1)
    u = torch.full((N,), float("-inf"), device=text.device).scatter_reduce_(0, g, t, reduce="amax")
    t2i = torch.empty(Q, dtype=torch.int64, device=text.device)
    i2t = torch.zeros(N, dtype=torch.int64, device=text.device)
    cols = torch.arange(N, device=text.device)
    step = max(1, chunk_bytes // (4 * N))
    for q0 in range(0, Q, step):
        q1 = min(Q, q0 + step)
        s = tn[q0:q1] @ xn.T
        neg = g[q0:q1, None] != cols[None, :]
        t2i[q0:q1] = ((s > t[q0:q1, None]) & neg).sum(1)
        i2t += ((s > u[None, :]) & neg).sum(0)
    has = torch.zeros(N, dtype=torch.bool, device=text.device)
    has[g] = True
    i2t[~has] = -1
    return t2i, i2t


def time_calls(fn, calls, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts), max(ts)


def kernel_ms(fn, reps=5):
    """Mean device time per call of the rank-count kernel (ares_kernel) from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.key_averages():
        if "ares_kernel" in ev.key:
            tot += getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
    return tot / reps / 1000.0


def band_check(got, ref, band):
    has = ref >= 0
    ok = bool(((got - ref).abs() <= band).all()) and bool(torch.equal(got < 0, ref < 0))
    return {"within_band": ok, "empty_band_fraction": (band[has] == 0).double().mean().item(),
            "exact_fraction": (got == ref).double().mean().item()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--sizes", default=",".join(SIZES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("retrieval_bench needs a CUDA device (B200)")
    import mae_clip_b200 as m
    from oracle import retrieval_eval_ref as R
    torch.backends.cuda.matmul.allow_tf32 = False
    result = {"gpu": gpu_info(), "D": D, "calls": args.calls, "sizes": []}
    for name in args.sizes.split(","):
        Q, N, per = SIZES[name]
        text, image, tti = make_inputs(Q, N, per, seed=Q + N)
        flop = 2.0 * Q * N * D
        row = {"name": name, "Q": Q, "N": N, "captions_per_image": per, "algorithmic_tflop": flop / 1e12}
        for mode in ("tc_f16x3", "tc_f16"):
            def call(mode=mode):
                return m.retrieval_ranks(text, image, tti, mode=mode)
            med, lo, hi = time_calls(call, args.calls)
            kms = kernel_ms(call)
            row[mode] = {"median_ms": med, "min_ms": lo, "max_ms": hi, "kernel_ms": kms,
                         "executed_tflops_over_kernel": PASSES[mode] * flop / (kms * 1e-3) / 1e12 if kms else None,
                         "algorithmic_tflops_over_call": flop / (med * 1e-3) / 1e12}
            print(name, mode, row[mode], flush=True)
        med, lo, hi = time_calls(lambda: torch_ranks(text, image, tti), args.calls, warmup=2)
        row["torch_fp32_chunked"] = {"median_ms": med, "min_ms": lo, "max_ms": hi,
                                     "algorithmic_tflops_over_call": flop / (med * 1e-3) / 1e12}
        row["speedup_tc_f16x3_vs_torch"] = med / row["tc_f16x3"]["median_ms"]
        print(name, "torch", row["torch_fp32_chunked"], flush=True)
        if Q * N <= 25000 * 5000:
            rt, ri, bt, bi = R.ranks_ref(text, image, tti, band=BAND["tc_f16x3"])
            _, _, bt16, bi16 = R.ranks_ref(text, image, tti, band=BAND["tc_f16"])
            parity = {}
            for mode, (b_t, b_i) in (("tc_f16x3", (bt, bi)), ("tc_f16", (bt16, bi16))):
                t2i, i2t = m.retrieval_ranks(text, image, tti, mode=mode)
                parity[mode] = {"text_to_image": band_check(t2i, rt, b_t), "image_to_text": band_check(i2t, ri, b_i),
                                "recall": m.retrieval_recall(text, image, tti, mode=mode)}
            tt2i, ti2t = torch_ranks(text, image, tti)
            parity["torch_fp32_chunked"] = {"text_to_image": band_check(tt2i, rt, bt),
                                            "image_to_text": band_check(ti2t, ri, bi)}
            parity["oracle_recall"] = R.recall_from_ranks(rt, ri)
            row["parity_vs_fp64"] = parity
            print(name, "parity", json.dumps(parity), flush=True)
        result["sizes"].append(row)
        del text, image, tti
        torch.cuda.empty_cache()
    js = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(js + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
