"""Where does rowgrad_kernel (the gradient row half, DESIGN 4.1) spend its time?  Times the row half of the stored-weights
gradient (mc_clip_bwd_rows: flagged-tile sweep + rowgrad_kernel + fold) at B = 32768 on each library given, per kernel
through torch.profiler, and reads the mbarrier wait counters of a -DMC_WAIT_PROFILE build.

Build the variants on any machine with nvcc (timing experiments only, results of the ablations are garbage):
    tools/build_variant.sh prof   -DMC_WAIT_PROFILE
    tools/build_variant.sh noepi  -DMC_ABLATE_EPI      (epilogue skips its arithmetic)
    tools/build_variant.sh nowst  -DMC_ABLATE_WSTORE   (the weights W are not written to global memory)
The -DMC_ABLATE_TMA build does not work with this tool: it also empties the rings of the pair_kernel sweeps that the
step runs, and at B = 32768 one of their ring producers stopped at a ring-slot barrier until the wait timed out and
trapped (cause not established).  The issuer's "ring slot full" share of the profile build measures the same thing.
Run (one GPU), each library in a process of its own, alternating over --rounds:
    python tools/rowgrad_profile.py [--rounds R] [--batch B] LIB...      (LIB "product" = mae_clip_b200/libmae_clip_b200.so)
Prints one JSON object: per library the median row-half ms, the median ms of every kernel of the row half, and, for a
profile build, each role's wait classes as a share of that role's lifetime (summed over the CTA pairs)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True

# slot -> name of rowgrad_kernel's wait classes (clip_loss_tc.cu, MC_WAIT_PROFILE); the first slot of a role is its lifetime
ROLES = {"issuer": (32, {33: "A rows", 34: "tile buffer free", 35: "ring slot full", 36: "weights", 37: "I_j^T tile",
                         38: "accumulator free"}),
         "ring producer": (40, {41: "job done", 42: "ring slot free"}),
         "I_j^T producer": (44, {45: "grad MMAs done"}),
         "epilogue h0": (48, {49: "constants", 50: "tile full", 51: "grad MMAs done", 52: "accumulator full",
                              53: "weight buffer stored"}),
         "epilogue h1": (56, {57: "constants", 58: "tile full", 59: "grad MMAs done", 60: "accumulator full",
                              61: "weight buffer stored"})}


def child(B, iters):
    import ctypes as C

    import torch
    sys.path.insert(0, ROOT)
    from bench import D_EMB, Phases, make_shard
    from mae_clip_b200 import _lib
    dev = torch.device("cuda", 0)
    ph = Phases(B, B, 0, "tc_f16x3", dev)
    I, T = make_shard(B, 1).to(dev), make_shard(B, 2).to(dev)
    ph.step(I, T)
    lib, ck, p, st = ph.lib, _lib.check, _lib.ptr, _lib.cur_stream()
    W = torch.empty(lib.mc_clip_stored_weights_bytes(B, B), device=dev, dtype=torch.uint8)
    diz = torch.zeros((B + 127) // 128 * 128, D_EMB, device=dev)
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)   # larger than L2: every call starts cold
    s = ph.stats_loc

    def rows():
        ck(lib.mc_clip_bwd_rows(p(ph.planes), B, B, D_EMB, 0, 1.0, ph.mode, p(s[0]), p(s[1]), p(s[2]), p(ph.gq_loc[0]),
                                p(ph.gq_loc[1]), None, p(ph.dT), p(diz), p(W), p(ph.flags), None, None, p(ph.ws),
                                ph.ws.numel(), st), "bwd_rows")

    raw = C.CDLL(_lib.LIB_PATH)
    prof = hasattr(raw, "mc_debug_wait_profile")
    if prof:
        raw.mc_debug_wait_profile.argtypes = [C.c_void_p, C.c_int]
    rows()
    torch.cuda.synchronize()
    if prof:
        assert raw.mc_debug_wait_profile(None, 1) == 0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = []
    for _ in range(iters):
        flush.fill_(1)
        ev[0].record()
        rows()
        ev[1].record()
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    out = {"rows_ms": statistics.median(ms), "rows_ms_all": [round(x, 4) for x in ms]}
    if prof:
        buf = (C.c_ulonglong * 64)()
        assert raw.mc_debug_wait_profile(buf, 1) == 0
        v = list(buf)
        out["waits"] = {role: {"lifetime_Mcycles_sum_over_pairs": round(v[tot] / 1e6, 2),
                               **{nm: round(v[t] / v[tot], 3) for t, nm in tags.items()}}
                        for role, (tot, tags) in ROLES.items() if v[tot]}
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as pr:
        for _ in range(iters):
            flush.fill_(1)
            rows()
        torch.cuda.synchronize()
    kern = {}
    for e in pr.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "fill" not in e.name and "elementwise" not in e.name:
            name = e.name.split("(")[0].replace("void mc::tc::", "")
            kern.setdefault(name, []).append(e.device_time / 1e3)
    out["kernels_ms"] = {k: round(statistics.median(v), 4) for k, v in kern.items()}
    print("RESULT " + json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.batch, a.iters)
        return
    res = {}
    for _ in range(a.rounds):
        for lib in a.libs:
            path = os.path.join(ROOT, "mae_clip_b200", "libmae_clip_b200.so") if lib == "product" else os.path.abspath(lib)
            env = dict(os.environ, MAE_CLIP_B200_LIB=path, PYTHONDONTWRITEBYTECODE="1")
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--batch", str(a.batch),
                                "--iters", str(a.iters), lib], env=env, capture_output=True, text=True, timeout=900)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
            if r.returncode != 0 or not line:
                raise RuntimeError(f"{lib}: exit {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
            res.setdefault(os.path.basename(lib), []).append(json.loads(line[0][7:]))
            print(f"{os.path.basename(lib)}: row half {res[os.path.basename(lib)][-1]['rows_ms']:.4f} ms", flush=True)
    summary = {}
    for lib, runs in res.items():
        summary[lib] = {"rows_ms_per_round": [round(x["rows_ms"], 4) for x in runs],
                        "kernels_ms": runs[-1]["kernels_ms"], **({"waits": runs[-1]["waits"]} if "waits" in runs[-1] else {})}
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
