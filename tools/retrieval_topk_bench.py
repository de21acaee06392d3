"""Retrieval top-k timing: mae_clip_b200.retrieval_topk (both tensor-core modes) against similarity_topk (fp32 SIMT,
full score matrix in the workspace) and the eager torch composition (F.normalize, fp32 matmul with TF32 off,
torch.topk; chunked over queries so that its score block stays within 4 GiB).

    python tools/retrieval_topk_bench.py [--calls 10] [--out FILE.json] [--shapes q1_1m,q1024_1m_k10,...]

Per shape and method: median of per-call CUDA-event times over `--calls` calls after one warm-up call of every method
of that shape; the workspace bytes the call needs (the eager composition: its largest score block plus the two
normalised copies); the algorithmic FLOPs 2QND and bytes (bank + queries read once, results written) and, for the
tensor-core modes, the executed tensor rate passes x 2QND / time.  D = 256, seeded random inputs.  The bank of the
1M shapes is 1 GiB, larger than the 126 MB L2, so it is read from HBM on every call.  The card's name, power limit and
maximum SM clock are read with nvidia-smi (a query only) in the same run and stored with the numbers.
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

D = 256
SHAPES = {  # name: (Q queries, N bank, k)
    "q1_1m": (1, 1 << 20, 10),
    "q1024_1m_k10": (1024, 1 << 20, 10),
    "q1024_1m_k100": (1024, 1 << 20, 100),
    "t2i_25k_5k": (25000, 5000, 10),
    "i2t_5k_25k": (5000, 25000, 10),
}
PASSES = {"tc_f16x3": 3, "tc_f16": 1}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"nvidia_smi": out}


def torch_topk(text, image, k, chunk_bytes=4 << 30):
    tn, xn = F.normalize(text, p=2, dim=-1), F.normalize(image, p=2, dim=-1)
    Q, N = tn.shape[0], xn.shape[0]
    step = max(1, chunk_bytes // (4 * N))
    vals, idx = [], []
    for q0 in range(0, Q, step):
        v, i = torch.topk(tn[q0:q0 + step] @ xn.T, k, dim=1)
        vals.append(v)
        idx.append(i)
    return torch.cat(vals), torch.cat(idx)


def torch_ws(Q, N, k, chunk_bytes=4 << 30):
    step = max(1, chunk_bytes // (4 * N))
    return 4 * min(Q, step) * N + 4 * (Q + N) * D


def time_calls(fn, calls):
    ts = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts), max(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("retrieval_topk_bench needs a CUDA device")
    import mae_clip_b200 as m
    from mae_clip_b200._lib import lib
    torch.backends.cuda.matmul.allow_tf32 = False
    result = {"gpu": gpu_info(), "D": D, "calls": args.calls, "shapes": {}}
    for name in args.shapes.split(","):
        Q, N, k = SHAPES[name]
        g = torch.Generator(device="cuda").manual_seed(Q + N + k)
        text = torch.randn(Q, D, device="cuda", generator=g)
        image = torch.randn(N, D, device="cuda", generator=g)
        flops = 2.0 * Q * N * D
        bytes_alg = 4.0 * (Q + N) * D + 12.0 * Q * k
        methods = {
            "retrieval_topk_tc_f16x3": (lambda: m.retrieval_topk(text, image, k, mode="tc_f16x3"),
                                        lib().mc_retrieval_topk_workspace_bytes(Q, N, D, k, 1)),
            "retrieval_topk_tc_f16": (lambda: m.retrieval_topk(text, image, k, mode="tc_f16"),
                                      lib().mc_retrieval_topk_workspace_bytes(Q, N, D, k, 2)),
            "similarity_topk": (lambda: m.similarity_topk(text, image, k),
                                lib().mc_similarity_topk_workspace_bytes(Q, N, D)),
            "torch_eager": (lambda: torch_topk(text, image, k), torch_ws(Q, N, k)),
        }
        for fn, _ in methods.values():   # warm every method of this shape first
            fn()
        torch.cuda.synchronize()
        ref_idx = m.retrieval_topk(text, image, k, mode="tc_f16x3")[1]
        row = {"Q": Q, "N": N, "k": k, "flops": flops, "bytes": bytes_alg, "methods": {}}
        for mname, (fn, ws) in methods.items():
            med, lo, hi = time_calls(fn, args.calls)
            r = {"ms_median": med, "ms_min": lo, "ms_max": hi, "workspace_bytes": int(ws),
                 "alg_tflops": flops / (med * 1e-3) / 1e12, "alg_hbm_gbs": bytes_alg / (med * 1e-3) / 1e9}
            for mode, passes in PASSES.items():
                if mname.endswith(mode):
                    r["executed_tensor_tflops"] = passes * flops / (med * 1e-3) / 1e12
            if mname != "retrieval_topk_tc_f16x3":
                idx = fn()[1]
                r["top1_agrees_with_tc_f16x3"] = (idx[:, 0] == ref_idx[:, 0]).double().mean().item()
            row["methods"][mname] = r
            print(name, mname, json.dumps(r), flush=True)
        result["shapes"][name] = row
        del text, image
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
