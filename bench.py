#!/usr/bin/env python
"""Benchmark of the mae_clip training-loss hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload c4|c2] [--mode tc_f16x3|tc_f16|simt_fp32] [--batch B] [--dump-outputs DIR]

Workload (BASELINE.json): the metric "contrastive+MAE loss fwd/bwd samples/s at 1/2/4/8 B200; % TC
/HBM roofline" is quoted on config 4, the global-batch contrastive loss at B = 32768, D = 256: it
is the only config that names 1..8 GPUs, it fits one B200 because no B x B tensor is ever
materialised, and the tensor-core roofline is only meaningful at that size (C2's B = 1024 is a
3.8 GFLOP, launch-bound problem).  The global batch is FIXED as N grows ("strong" scaling): rank r
owns rows [r B/N, (r+1) B/N).  A step = one forward + backward of the loss over the whole global
batch from fp32 embeddings already in HBM: stage operands, row/col statistics sweep, row-loss
sweep, gradient sweep.  When N > 1 the exchange steps run over mapped peer memory by default
(--transport peer: the embedding all-gather is fused into the operand staging, statistics are pushed
by our own kernels; --transport nccl keeps the torch.distributed all-gathers).  At N = 1 the line also carries the C2
latency and C5 MAE numbers under "extra".

e2e is the same step through the C-ABI entry point that takes HOST buffers
(mc_clip_loss_fwd_bwd_host at N = 1; pinned-host shards -> H2D -> dist loss -> D2H at N > 1).

--impl reference times the reference's own CPU implementation of the path (the op-for-op oracle
port of CLIP.py:34-43 + autograd; the Python reference cannot travel to the GPU box) with all host
threads on a bounded sample; see cpu_baseline.sample.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # a run writes nothing into the tree, which may be read-only

D_EMB = 256
DUMP_ROWS = 16384   # --dump-outputs: rows of dI / dT written, a fixed sample when a rank owns more (32 MiB in all)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c2"])
    ap.add_argument("--mode", default="auto")
    ap.add_argument("--batch", type=int, default=0, help="global batch (default: 32768 for c4, 1024 for c2)")
    ap.add_argument("--cpu-sample-batch", type=int, default=0,
                    help="rows of the bounded CPU sample (0 = the largest power of two <= 16384 whose ~20 B x B fp32 "
                         "temporaries fit the host's free RAM: 21 GiB at 16384, 5 GiB at 8192)")
    ap.add_argument("--transport", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: peer = our kernels over mapped peer memory (default), nccl = torch.distributed all-gathers")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the global batch stays 32768 as N grows; weak: 4096 rows per GPU, B = 4096 N "
                         "(config 4 read literally; the loss is O(B^2), so samples/s per GPU then FALLS with N by construction)")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as float32 DIR/<name>.npy: loss, and "
                         "dI / dT (rank 0's rows; above %d rows the rows np.random.RandomState(0).choice(rows, %d, "
                         "replace=False) in ascending order)" % (DUMP_ROWS, DUMP_ROWS))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    return args


# ------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
            # nvidia-smi needs a few hundred ms before its first sample: wait for it, or the whole (sub-second) run
            # is over before the sampler sees anything
            t0 = time.perf_counter()
            while not self.lines and time.perf_counter() - t0 < 5.0 and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def make_shard(b, seed, scale=1.0):
    """Embeddings with the distribution ProjectionHead emits (LayerNorm'd gaussian rows)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, D_EMB, generator=g)
    return torch.nn.functional.layer_norm(x, (D_EMB,)) * scale


def cpu_sample_batch(args, B_work):
    """Largest power-of-two sample batch the host can hold: the reference materialises ~20 B x B fp32 tensors (forward
    temporaries + what autograd keeps), i.e. ~21 GiB at B = 16384 and ~5.4 GiB at 8192."""
    Bs = min(args.cpu_sample_batch, B_work) if args.cpu_sample_batch else B_work
    if not args.cpu_sample_batch:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 8 << 30
        Bs = min(B_work, 16384)
        while Bs > 1024 and 20 * Bs * Bs * 4 * 1.5 > avail:
            Bs //= 2
        # keep the whole CPU leg within ~2 minutes: ~8 s per step at B = 16384 on 16 cores, O(B^2)
        n_steps = max(1, getattr(args, "_cpu_steps", 3))
        while Bs > 2048 and n_steps * 8.0 * (Bs / 16384.0) ** 2 * (16.0 / max(1, os.cpu_count() or 1)) > 120.0:
            Bs //= 2
    return Bs


def cpu_reference_leg(args, B_work, steps, warmup):
    """The oracle port of the reference loss (CLIP.py:34-43 + autograd) on host cores."""
    import torch

    from oracle import loss_ref
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    args._cpu_steps = steps + warmup
    Bs = cpu_sample_batch(args, B_work)
    I = make_shard(Bs, 0)
    T = make_shard(Bs, 1)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss_ref.clip_loss_fwd_bwd_ref(I, T, 1.0)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    raw = Bs / t
    # cost per sample is linear in B (the loss is O(B^2 D)): project the sample to the workload's B
    value = raw * (Bs / B_work)
    sample = (f"MEASURED: full reference loss fwd+bwd (oracle port, torch CPU fp32, {cores} threads) at B={Bs}: "
              f"{t * 1e3:.1f} ms/step = {raw:.0f} samples/s at that B (the largest batch whose ~20 B x B fp32 temporaries fit "
              f"this host's RAM); PROJECTED to the workload's B={B_work} by the O(B^2) cost (x {Bs}/{B_work}): "
              f"{value:.0f} samples/s") if Bs != B_work else \
             (f"MEASURED: full reference loss fwd+bwd (oracle port, torch CPU fp32, {cores} threads) at B={Bs}: "
              f"{t * 1e3:.1f} ms/step")
    return {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample,
            "ms_per_sample_step": t * 1e3, "sample_batch": Bs, "measured_samples_per_s_at_sample_batch": raw,
            "projected": Bs != B_work}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.batch or (32768 if args.workload == "c4" else 1024)
    steps, warmup = max(1, args.steps), max(0, args.warmup)  # exactly K timed steps after W warm-ups
    cb = cpu_reference_leg(args, B, steps, warmup)
    line = {"impl": "reference", "metric": "contrastive loss fwd+bwd samples/s", "value": cb["value"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": cb["ms_per_sample_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args, B, "cpu"),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_batch",
                                                "measured_samples_per_s_at_sample_batch", "projected")},
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(args, B, mode):
    name = ("c4: global-batch contrastive soft-target loss fwd+bwd, B=%d D=%d, rows sharded over ranks" % (B, D_EMB)
            if args.workload == "c4" else
            "c2: CLIP loss-only microbench fwd+bwd, B=%d D=%d fp32" % (B, D_EMB))
    return {"workload": name, "global_batch": B, "dim": D_EMB, "temperature": 1.0, "engine": mode,
            "parallelism": f"row-sharded x{args.gpus}", "l2": "flushed between timed steps (256 MiB write)"}


# ------------------------------------------------------------------------------------------------
def pick_mode(args):
    from mae_clip_b200 import _lib
    if args.mode != "auto":
        return args.mode
    return "tc_f16x3" if _lib.lib().mc_clip_planes_bytes(128, D_EMB, _lib.GEMM_MODES["tc_f16x3"]) > 256 \
        else "simt_fp32"


class Phases:
    """One step on one rank through the C ABI, with CUDA events between the phases so the dominant
    kernel's duration is measured live on the launching stream."""

    def __init__(self, B, b, row_offset, mode, device, sparse=None):
        import torch

        from mae_clip_b200 import _lib
        self.torch, self._lib, self.lib = torch, _lib, _lib.lib()
        self.B, self.b, self.off, self.mode = B, b, row_offset, _lib.GEMM_MODES[mode]
        f32 = dict(device=device, dtype=torch.float32)
        self.stats_loc = torch.empty(4, b, **f32)  # r, c, rz, sum_j P_ij S_ij
        self.gq_loc = torch.empty(2, b, **f32)
        self.part = torch.empty(1, **f32)
        self.part_buf = self.part
        self.pack = torch.zeros(3, b, **f32)
        self.dI = torch.empty(b, D_EMB, **f32)
        self.dT = torch.empty(b, D_EMB, **f32)
        nb = self.lib.mc_clip_planes_bytes(B, D_EMB, self.mode)
        self.planes = torch.empty(max(nb, 1), device=device, dtype=torch.uint8)
        if sparse is None:
            sparse = os.environ.get("MAE_CLIP_DENSE", "0") != "1"
        nf = self.lib.mc_clip_tile_flags_bytes(b, B, D_EMB, self.mode) if sparse else 0
        self.flags_raw = torch.empty(nf, device=device, dtype=torch.uint8) if nf else None
        self.flags = torch.empty(nf, device=device, dtype=torch.uint8) if nf else None
        nws = self.lib.mc_clip_loss_workspace_bytes(b, B, D_EMB, self.mode)
        self.ws = torch.empty(max(nws, 1), device=device, dtype=torch.uint8)
        self.ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]

    def step(self, I_all, T_all, gather_vec=None, record=False):
        lib, ck, p = self.lib, self._lib.check, self._lib.ptr
        st = self._lib.cur_stream()
        B, b, off, mode = self.B, self.b, self.off, self.mode
        ev = self.ev
        if record: ev[0].record()
        ck(lib.mc_clip_prepare(p(I_all), p(T_all), B, B, D_EMB, 0, mode, p(self.planes), st), "prepare")
        if record: ev[1].record()
        ck(lib.mc_clip_stats(p(I_all), p(T_all), p(self.planes), b, B, D_EMB, off, 1.0, mode, p(self.stats_loc[0]),
                             p(self.stats_loc[1]), p(self.stats_loc[2]), p(self.stats_loc[3]), p(self.flags_raw), p(self.ws),
                             self.ws.numel(), st), "stats")
        stats_all = gather_vec(self.stats_loc[:3]) if gather_vec else self.stats_loc
        if self.flags_raw is not None:   # tile flags: gather the raw bitmap rows of every rank, OR in the transpose
            flags_all = self.flags_raw
            if gather_vec:
                import torch.distributed as dist
                flags_all = self.torch.empty(self.flags_raw.numel() * (B // b), device=self.flags_raw.device, dtype=self.torch.uint8)
                dist.all_gather_into_tensor(flags_all, self.flags_raw)
            ck(lib.mc_clip_flags_finalize(p(flags_all), B, b, off, p(self.flags), st), "flags_finalize")
        if record: ev[2].record()
        ck(lib.mc_clip_rowloss(p(I_all), p(T_all), p(self.planes), b, B, D_EMB, off, 1.0, mode, p(stats_all[0]),
                               p(stats_all[1]), p(stats_all[2]), p(self.stats_loc[3]), p(self.gq_loc[0]), p(self.gq_loc[1]), p(self.part_buf),
                               p(self.flags), p(self.ws), self.ws.numel(), st), "rowloss")
        if gather_vec:  # the loss partial rides along with the two vectors: one collective instead of two
            self.pack[:2] = self.gq_loc
            self.pack[2, 0:1] = self.part_buf
            g3 = gather_vec(self.pack)
            gq_all = g3[:2]
            self.part = g3[2].reshape(-1, self.b)[:, 0].sum().reshape(1)
        else:
            gq_all = self.gq_loc
        if record: ev[3].record()
        ck(lib.mc_clip_bwd(p(I_all), p(T_all), p(self.planes), b, B, D_EMB, off, 1.0, mode, p(stats_all[0]),
                           p(stats_all[1]), p(stats_all[2]), p(gq_all[0]), p(gq_all[1]), None, p(self.dI), p(self.dT),
                           p(self.flags), p(self.ws), self.ws.numel(), st), "bwd")
        if record: ev[4].record()
        return self.part

    def phase_ms(self):
        e = self.ev
        return [e[i].elapsed_time(e[i + 1]) for i in range(4)]


class PeerPhases:
    """Same step over the peer-memory transport (mae_clip_b200/dist.py PeerStep): every exchange is a
    kernel of libmae_clip_b200.so on this stream; the embedding all-gather is fused into the staging."""

    def __init__(self, B, b, rank, mode, device):
        from mae_clip_b200.dist import PeerStep
        from mae_clip_b200.peer import get_exchange
        self.step_impl = PeerStep(get_exchange(b, D_EMB), mode)
        self.part = self.dI = self.dT = None
        self.ev = []

    def step(self, I_loc, T_loc, record=False):
        ev = [] if record else None
        loss, saved = self.step_impl.forward(I_loc, T_loc, 1.0, ev)
        self.last_flags = saved[2]
        self.dI, self.dT = self.step_impl.backward(saved, 1.0, None, ev)
        self.part = loss.reshape(1)
        if record:
            self.ev = ev
        return self.part

    def phase_ms(self):
        e = self.ev  # start, staged, stats exchanged, row loss exchanged, gradients
        return [e[i].elapsed_time(e[i + 1]) for i in range(4)]


def run_b200(args):
    import torch
    import torch.distributed as dist

    from mae_clip_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    B = args.batch or (32768 if args.workload == "c4" else 1024)
    if args.scaling == "weak":
        B = (args.batch or 4096) * world
    assert B % world == 0
    b = B // world
    mode = pick_mode(args)
    lib = _lib.lib()
    peaks = load_peaks()

    # this rank's shard; C4 seeds 1000 + r per 4096-row block so the global batch is the same for every N
    blk = 4096 if B % 4096 == 0 and b % 4096 == 0 else b
    shard_I = torch.cat([make_shard(blk, 1000 + (rank * b) // blk + i) for i in range(b // blk)])
    shard_T = torch.cat([make_shard(blk, 5000 + (rank * b) // blk + i) for i in range(b // blk)])
    host_I, host_T = shard_I.pin_memory(), shard_T.pin_memory()
    I_loc, T_loc = host_I.to(dev), host_T.to(dev)

    def gather_rows(x):  # (b, D) per rank -> (B, D)
        if world == 1:
            return x
        out = torch.empty(world * x.shape[0], x.shape[1], device=dev, dtype=x.dtype)
        dist.all_gather_into_tensor(out, x)
        return out

    def gather_vec(x):  # (k, b) per rank -> (k, B)
        k = x.shape[0]
        buf = torch.empty(world, k, b, device=dev, dtype=x.dtype)
        dist.all_gather_into_tensor(buf.view(-1), x.contiguous().view(-1))
        return buf.permute(1, 0, 2).reshape(k, B).contiguous()

    transport = args.transport
    if transport == "auto":
        transport = "peer" if (world > 1 and mode != "simt_fp32" and b % 128 == 0) else "nccl"
    if world == 1:
        transport = "none"
    ph = None
    if transport == "peer":
        from mae_clip_b200.peer import PeerUnavailable
        try:
            ph = PeerPhases(B, b, rank, mode, dev)
        except PeerUnavailable as e:  # raised on every rank together (no P2P / IPC on this box)
            if args.transport == "peer":
                raise
            if rank == 0:
                print(f"bench: peer memory unavailable ({e}); using the NCCL transport", file=sys.stderr)
            transport = "nccl"
    if ph is None:
        ph = Phases(B, b, rank * b, mode, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def one_step(record=False, I=None, T=None):
        I, T = (I_loc if I is None else I), (T_loc if T is None else T)
        if transport == "peer":
            return ph.step(I, T, record=record)
        I_all, T_all = gather_rows(I), gather_rows(T)
        return ph.step(I_all, T_all, gather_vec if world > 1 else None, record=record)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from the warm-up on (same workload): the timed region of a sharded run is only tens of ms
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()

    # N > 1, peer transport: the whole step (push, barriers, staging, three sweeps, finalize kernels - ~25 launches of our
    # library, no collective-library call) is captured ONCE in a CUDA graph and replayed: at 4096 rows per rank the step
    # is ~1.2 ms and the per-launch gaps were a fifth of it.  The peer barrier keeps its epoch in device memory for this.
    graph, launches_per_step = None, None
    phase_ms_eager = [0.0] * 4
    # N = 1: the same capture (22 launches of our library, no host sync inside the step); the gaps between the short
    # finalize/staging kernels are ~1% of the step.
    if (transport == "peer" or world == 1) and os.environ.get("MAE_CLIP_BENCH_GRAPH", "1") != "0":
        for _ in range(args.steps):            # per-phase times from eager steps (events cannot sit inside the replayed graph)
            flush.fill_(1)
            barrier()
            one_step(record=True)
            barrier()
            for i, v in enumerate(ph.phase_ms()):
                phase_ms_eager[i] += v
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                one_step()                      # allocations of the capture stream's workspace happen here
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            g = torch.cuda.CUDAGraph()
            n0 = lib.mc_kernel_launch_count()
            with torch.cuda.graph(g, stream=side):
                one_step()
            launches_per_step = int(lib.mc_kernel_launch_count() - n0)
            graph = g
            barrier()
            for _ in range(2):
                graph.replay()
            barrier()
        except Exception as e:  # noqa: BLE001 - capture is an optimisation: fall back to eager launches, say so
            if rank == 0:
                print(f"bench: CUDA graph capture of the step failed ({type(e).__name__}: {e}); eager launches", file=sys.stderr)
            graph = None
        if world > 1:
            ok = torch.tensor([1 if graph is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)       # every rank replays, or none does
            if not ok.item():
                graph = None

    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.mc_kernel_launch_count()
    total_ms, phase_ms = 0.0, [0.0] * 4
    for _ in range(args.steps):
        flush.fill_(1)  # evict L2 between timed iterations (outside the timed region)
        barrier()
        t_start.record()
        if graph is not None:
            graph.replay()
        else:
            one_step(record=True)
        t_end.record()
        barrier()
        total_ms += t_start.elapsed_time(t_end)
        if graph is None:
            for i, v in enumerate(ph.phase_ms()):
                phase_ms[i] += v
    launches = lib.mc_kernel_launch_count() - launches0
    if graph is not None:
        launches = launches_per_step * args.steps
        phase_ms = phase_ms_eager
    if args.dump_outputs and rank == 0:   # before anything else reuses the step's buffers
        dump_outputs(args.dump_outputs, ph)
    loss_val = float(ph.part.item())
    tmax = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = tmax.item()
    ms_per_step = total_ms / args.steps
    value = B / (ms_per_step * 1e-3)

    # ---- parity of THIS run's numbers (N > 1): every rank rebuilds the global batch from the seeds, runs the single-GPU
    # fused step on it and compares its shard of the sharded step with it (outside the timed region); rank 0 also checks
    # its shard against the fp64 blockwise oracle (checker only)
    parity = None
    if world > 1:
        nblk = B // blk
        I_full = torch.cat([make_shard(blk, 1000 + k) for k in range(nblk)]).to(dev)
        T_full = torch.cat([make_shard(blk, 5000 + k) for k in range(nblk)]).to(dev)
        md = _lib.GEMM_MODES[mode]
        nws = lib.mc_clip_loss_fused_workspace_bytes(B, D_EMB, md)
        fws = torch.empty(nws, dtype=torch.uint8, device=dev)
        l1, dI1, dT1 = torch.zeros(1, device=dev), torch.empty_like(I_full), torch.empty_like(T_full)
        _lib.check(lib.mc_clip_loss_fwd_bwd(I_full.data_ptr(), T_full.data_ptr(), B, D_EMB, 1.0, md, l1.data_ptr(),
                                            dI1.data_ptr(), dT1.data_ptr(), fws.data_ptr(), nws, _lib.cur_stream()),
                   "mc_clip_loss_fwd_bwd (parity)")
        rows = slice(rank * b, (rank + 1) * b)

        def rel(a, r):
            return ((a.double() - r.double()).norm() / r.double().norm()).item()
        pv = [abs(loss_val - l1.item()) / abs(l1.item()), rel(ph.dI, dI1[rows]), rel(ph.dT, dT1[rows])]
        if rank == 0:
            from oracle import loss_blockwise
            ol, odI, odT, _ = loss_blockwise.clip_loss_blockwise_f64(I_full, T_full, 1.0, rows=1024)
            pv += [abs(loss_val - ol) / abs(ol), rel(ph.dI, odI[rows]), rel(ph.dT, odT[rows])]
            del odI, odT
        else:
            pv += [0.0, 0.0, 0.0]
        pt = torch.tensor(pv, device=dev, dtype=torch.float64)
        dist.all_reduce(pt, op=dist.ReduceOp.MAX)
        pv = pt.tolist()
        parity = {"vs": "single-GPU fused step on the same global batch, max over ranks", "loss_rel": pv[0], "dI_rel": pv[1],
                  "dT_rel": pv[2], "rank0_shard_vs_fp64_oracle": {"loss_rel": pv[3], "dI_rel": pv[4], "dT_rel": pv[5]},
                  "tolerance": "loss 1e-4, gradients 1e-3 relative (north_star)"}
        del I_full, T_full, dI1, dT1, fws

    # ---- e2e: host buffers in, loss + gradients out, copies inside the timed region
    e2e_ms = 0.0
    h2d = 2 * b * D_EMB * 4
    d2h = 2 * b * D_EMB * 4 + 4
    if world == 1:
        nws = lib.mc_clip_loss_host_workspace_bytes(B, D_EMB, _lib.GEMM_MODES[mode])
        dws = torch.empty(nws, dtype=torch.uint8, device=dev)
        out_dI, out_dT = torch.empty_like(host_I).pin_memory(), torch.empty_like(host_T).pin_memory()
        out_loss = torch.zeros(1).pin_memory()
        st = torch.cuda.current_stream().cuda_stream

        def e2e_step():
            _lib.check(lib.mc_clip_loss_fwd_bwd_host(host_I.data_ptr(), host_T.data_ptr(), B, D_EMB, 1.0,
                                                     _lib.GEMM_MODES[mode], out_loss.data_ptr(), out_dI.data_ptr(),
                                                     out_dT.data_ptr(), dws.data_ptr(), nws, ctypes.c_void_p(st)),
                       "mc_clip_loss_fwd_bwd_host")
    else:
        out_dI, out_dT = torch.empty_like(host_I).pin_memory(), torch.empty_like(host_T).pin_memory()
        out_loss = torch.zeros(1).pin_memory()

        def e2e_step():
            # pinned host shards -> the step's input buffers, the (graph-replayed) step, gradients + loss back to pinned host
            I_loc.copy_(host_I, non_blocking=True)
            T_loc.copy_(host_T, non_blocking=True)
            if graph is not None:
                graph.replay()
                part = ph.part
            else:
                part = one_step(False)
            out_dI.copy_(ph.dI, non_blocking=True)
            out_dT.copy_(ph.dT, non_blocking=True)
            out_loss.copy_(part, non_blocking=True)
            torch.cuda.current_stream().synchronize()

    e2e_step()
    e_steps = args.steps
    for _ in range(e_steps):
        flush.fill_(1)
        barrier()
        t0 = time.perf_counter()
        e2e_step()
        torch.cuda.synchronize()
        e2e_ms += (time.perf_counter() - t0) * 1e3
    emax = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(emax, op=dist.ReduceOp.MAX)
    e2e_value = B / (emax.item() / e_steps * 1e-3)
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        flops_step = 14.0 * B * B * D_EMB / world          # algorithmic, this rank's strip
        bwd_ms = phase_ms[3] / args.steps
        flops_bwd = 8.0 * B * B * D_EMB / world            # the gradient sweep: 4 GEMMs (SURVEY 8d)
        achieved = flops_bwd / (bwd_ms * 1e-3) / 1e12
        # which peak: the burst figure when the SM clock sat at (>= 95% of) its maximum during the run - a kernel timed
        # alone for milliseconds - else the sustained one
        at_max_clock = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and
                            clocks["sm_mhz"] >= 0.95 * clocks["sm_max_mhz"])
        peak_kind = "burst" if (at_max_clock or not peaks["tc_sustained"]) else "sustained"
        peak = peaks["tc_burst"] if peak_kind == "burst" else peaks["tc_sustained"]
        # executed tensor-core work of the gradient sweep, in GEMM units of 2 B^2 D / world FLOPs: S and S^T recomputed
        # (2 units x passes) + their two gradient GEMMs, and - only on the tiles flagged as carrying soft-target mass -
        # Z (2 units x passes, K = 2D) + the two dZ GEMMs.  The algorithmic count (SURVEY 8d) is the 4 gradient GEMMs.
        passes = 3 if mode == "tc_f16x3" else 1
        flags_t = getattr(ph, "flags", None)
        if flags_t is None and hasattr(ph, "step_impl"):
            flags_t = getattr(ph, "last_flags", None)
        density = float(flags_t.float().mean().item()) if flags_t is not None else 1.0
        # which form of the gradient ran: a call that owns every row (one GPU) and the peer transport's default take
        # the STORED-WEIGHTS form - S once (passes) + dT GEMM in the row half, dI from the stored fp16 weights in the
        # column half (1 unit), and on the flagged tiles only the soft-target part: the split form recomputes S, S^T, Z
        # (K = 2D) there and runs four small GEMMs, the single sweep (no flags / MAE_CLIP_BWD_SPLIT=0) adds S^T, Z and the
        # two dZ GEMMs to its own S; the OWN-ROWS form recomputes the transposed strip everywhere instead of storing
        form = "ownrows"
        if mode != "simt_fp32" and os.environ.get("MAE_CLIP_BWD_FORM") != "ownrows":
            if world == 1 or (transport == "peer" and getattr(ph.step_impl, "bwd_form", "") == "stored"):
                form = "stored"
        if form == "stored" and flags_t is not None and density > GATE_DENSITY:
            form = "ownrows"    # the device-side gate (mc_clip_bwd_gate) chose the own-rows kernels for this batch
        split = form == "stored" and flags_t is not None and mode == "tc_f16x3" and os.environ.get("MAE_CLIP_BWD_SPLIT") != "0"
        if mode == "simt_fp32":
            exec_units = 8
        elif form == "stored":
            exec_units = (passes + 1) + 1 + density * ((4 * passes + 4) if split else (3 * passes + 2))
        else:
            exec_units = (2 * passes + 2) + density * (2 * passes + 2)
        executed = exec_units * 2.0 * B * B * D_EMB / world / (bwd_ms * 1e-3) / 1e12
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "r02_roofline_ncu.json")))
        except Exception:
            pass
        traffic_ok = bool(ncu) and mode == "tc_f16x3" and world == 1 and B == 32768
        line = {
            "metric": "contrastive loss fwd+bwd samples/s", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": {"simt_fp32": "fp32", "tc_f16x3": "fp32 (fp16 hi+lo split operands, 3 tcgen05 passes, fp32 accumulate)",
                      "tc_f16": "fp16 operands, fp32 accumulate"}[mode],
            "data": "synthetic", "config": dict(workload_config(args, B, mode), transport=(
                transport + "-" + ph.step_impl.exchange_mode if transport == "peer" else transport),
                launch=("one CUDA graph replay per step" if graph is not None else "eager launches"),
                soft_target_tiles=("every tile (dense)" if flags_t is None else
                                   "flagged tiles only: %.4f of the %d x %d tiles can hold P_ij >= 2^-44" % (
                                       density, flags_t.numel() // ((B + 127) // 128), (B + 127) // 128))), "loss": loss_val,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "ms_per_step": emax.item() / e_steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "phases_ms": {"prepare": phase_ms[0] / args.steps, "stats": phase_ms[1] / args.steps,
                          "rowloss": phase_ms[2] / args.steps, "bwd": bwd_ms,
                          "timed": "eager steps with events between the phases" + (
                              " (the headline ms_per_step is the graph replay)" if graph is not None else "")},
            "roofline": {"bound": "tensor",
                         "kernel": "gradient phase (mc_clip_bwd): " + {
                             "stored": ("rowgrad_kernel + flagged-tile sweep + colgrad_kernel" if split else
                                        "row sweep (stores the fp16 weights) + colgrad_kernel"),
                             "ownrows": "own-rows sweep (transposed strip recomputed)"}[form],
                         "gradient_form": form, "achieved": achieved,
                         "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "peak_source": "%s, bf16 %s (fp16 runs at the same tensor rate); the SM clock %s during the run" % (
                             peaks["source"], peak_kind, "sat at its maximum" if at_max_clock else "was below 95% of its maximum"),
                         "frac_vs_burst": achieved / peaks["tc_burst"],
                         "frac_vs_sustained": achieved / (peaks["tc_sustained"] or peaks["tc_burst"]),
                         # DRAM bytes of ONE gradient-sweep launch from the committed ncu --set full capture of this
                         # round (not measured in this run; null when this run is not that configuration)
                         "traffic": ncu.get("traffic_bytes_per_launch") if traffic_ok else None,
                         "traffic_source": ncu.get("source") if traffic_ok else None,
                         "executed_tflops": executed, "executed_frac": executed / peak,
                         "executed_gemm_units": exec_units, "algorithmic_gemm_units": 4,
                         "frac_ceiling_note": "the %s form executes %.2f GEMM units per 4 algorithmic ones: frac <= %.2f "
                                              "at 100%% of the tensor peak" % (form, exec_units, 4.0 / exec_units),
                         # the other tensor-bound kernel of the step: the statistics sweep (S in 3 passes + the hi-plane
                         # probe of Z, K = 2D; algorithmic forward work 6 B^2 D: S, I I^T, T T^T)
                         "stats_sweep": {"ms": phase_ms[1] / args.steps,
                                         "achieved": 6.0 * B * B * D_EMB / world / (phase_ms[1] / args.steps * 1e-3) / 1e12,
                                         "frac": 6.0 * B * B * D_EMB / world / (phase_ms[1] / args.steps * 1e-3) / 1e12 / peak},
                         "tile_flag_density": density,
                         "algorithmic_flops_per_launch": flops_bwd,
                         "step_achieved": flops_step / (ms_per_step * 1e-3) / 1e12,
                         "step_frac": flops_step / (ms_per_step * 1e-3) / 1e12 / peak},
        }
        if parity is not None:
            line["parity"] = parity
        if world == 1 and mode != "simt_fp32" and not args.no_extra:
            # the two regimes the tile flags separate, measured in this run: every tile computed (flags off), and the
            # soft-target regime (embeddings x 0.25: every tile carries mass, flag density 1.0, flags on)
            try:
                line["roofline"]["gradient_halves"] = gradient_halves(ph, B, mode, flush, peak)
            except Exception as e:  # noqa: BLE001 - context only
                line["roofline"]["gradient_halves"] = {"error": f"{type(e).__name__}: {e}"}
            line["roofline"]["dense"] = regime(B, mode, dev, flush, I_loc, T_loc, False, peak, peaks)
            line["roofline"]["soft"] = regime(B, mode, dev, flush, I_loc * 0.25, T_loc * 0.25, True, peak, peaks)
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_reference_leg(args, B, 2, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_batch",
                                                       "measured_samples_per_s_at_sample_batch", "projected")}
        if not args.no_extra and world == 1:
            line["extra"] = extras(dev, mode, peaks, peak)
            if mode == "tc_f16x3":
                line["extra"].update(single_pass_context(B, I_loc, T_loc, dev, flush, peaks, peak))
            line["extra"].update(reference_formulation_gpu(B, I_loc, T_loc, ms_per_step))
        print(json.dumps(line))
    if world > 1:
        if transport == "peer":
            from mae_clip_b200 import peer
            peer.close_all()
        dist.destroy_process_group()


def dump_outputs(out_dir, ph):
    """--dump-outputs: the loss and this rank's gradients dI / dT as the last timed step left them.  The inputs are
    seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    b = ph.dI.shape[0]
    rows = np.arange(b)
    if b > DUMP_ROWS:
        rows = np.sort(np.random.RandomState(0).choice(b, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(ph.dI.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", ph.part.reshape(())), ("dI", ph.dI.index_select(0, idx)), ("dT", ph.dT.index_select(0, idx))):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def gradient_halves(ph, B, mode, flush, peak):
    """The two halves of the stored-weights gradient timed separately with CUDA events through their own C-ABI entry
    points, on the statistics the last timed step left in `ph` (one GPU): the row half is the flagged-tile sweep +
    rowgrad_kernel + fold (S in 3 passes + the dT GEMM: 4 GEMM units), the column half colgrad_kernel + fold (1 unit,
    bound by the 2 B^2 bytes of fp16 weights it reads)."""
    import torch
    lib, ck, p = ph.lib, ph._lib.check, ph._lib.ptr
    if ph.flags is None or B * B < 4096 * 4096:
        return None
    dev = ph.dI.device
    md = ph.mode
    W = torch.empty(lib.mc_clip_stored_weights_bytes(B, B), device=dev, dtype=torch.uint8)
    diz = torch.zeros((B + 127) // 128 * 128, D_EMB, device=dev)
    wsc = torch.empty(lib.mc_clip_bwd_cols_workspace_bytes(B, D_EMB), device=dev, dtype=torch.uint8)
    st = ph._lib.cur_stream()
    s = ph.stats_loc
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    rows_ms = cols_ms = 0.0
    n = 5
    for it in range(n + 2):
        flush.fill_(1)
        torch.cuda.synchronize()
        ev[0].record()
        ck(lib.mc_clip_bwd_rows(p(ph.planes), B, B, D_EMB, 0, 1.0, md, p(s[0]), p(s[1]), p(s[2]), p(ph.gq_loc[0]), p(ph.gq_loc[1]),
                                None, p(ph.dT), p(diz), p(W), p(ph.flags), None, None, p(ph.ws), ph.ws.numel(), st), "bwd_rows")
        ev[1].record()
        ck(lib.mc_clip_bwd_cols(p(ph.planes), B, D_EMB, 1.0, md, p(s[0]), p(s[1]), p(s[2]), p(ph.gq_loc[1]), None, p(W), B, 0, 0, B,
                                p(diz), p(ph.dI), None, p(wsc), wsc.numel(), st), "bwd_cols")
        ev[2].record()
        torch.cuda.synchronize()
        if it >= 2:
            rows_ms += ev[0].elapsed_time(ev[1]) / n
            cols_ms += ev[1].elapsed_time(ev[2]) / n
    unit = 2.0 * B * B * D_EMB / 1e12
    passes = 3 if md == 1 else 1
    return {"rows_ms": rows_ms, "cols_ms": cols_ms,
            "rows_executed_TFLOPs": (passes + 1) * unit / (rows_ms * 1e-3), "rows_executed_frac": (passes + 1) * unit / (rows_ms * 1e-3) / peak,
            "cols_executed_TFLOPs": unit / (cols_ms * 1e-3), "cols_GBps_weights_read": 2.0 * B * B / (cols_ms * 1e-3) / 1e9,
            "note": "row half = flagged-tile sweep + rowgrad_kernel + fold (executed: S x passes + dT GEMM); column half = "
                    "colgrad_kernel + fold (HBM-bound on the stored fp16 weights)"}


GATE_DENSITY = 0.15   # mc_clip_bwd_gate: the stored-weights gradient runs iff the tile-flag density is at most this


def regime(B, mode, dev, flush, I, T, sparse, peak, peaks):
    """The same step in another soft-target regime (see run_b200): ms per step and the gradient sweep's roofline terms."""
    import torch
    ph = Phases(B, B, 0, mode, dev, sparse=sparse)
    for _ in range(2):
        ph.step(I, T)
    torch.cuda.synchronize()
    n, tot, phs = 3, 0.0, [0.0] * 4
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(n):
        flush.fill_(1)
        torch.cuda.synchronize()
        a.record()
        ph.step(I, T, record=True)
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
        for i, v in enumerate(ph.phase_ms()):
            phs[i] += v
    ms, bwd_ms = tot / n, phs[3] / n
    density = float(ph.flags.float().mean().item()) if ph.flags is not None else 1.0
    passes = 3 if mode == "tc_f16x3" else 1
    gated_out = ph.flags is not None and density > GATE_DENSITY   # the device-side gate picks the own-rows kernels
    if mode == "simt_fp32" or os.environ.get("MAE_CLIP_BWD_FORM") == "ownrows" or gated_out:
        units = (2 * passes + 2) * (1 + density)
    else:   # stored-weights form (see run_b200): split when tile flags exist, the single row sweep otherwise
        split = sparse and mode == "tc_f16x3" and os.environ.get("MAE_CLIP_BWD_SPLIT") != "0"
        units = (passes + 1) + 1 + density * ((4 * passes + 4) if split else (3 * passes + 2))
    ach = 8.0 * B * B * D_EMB / (bwd_ms * 1e-3) / 1e12
    return {"ms_per_step": ms, "samples_per_s": B / (ms * 1e-3), "loss": float(ph.part.item()),
            "phases_ms": {"prepare": phs[0] / n, "stats": phs[1] / n, "rowloss": phs[2] / n, "bwd": bwd_ms},
            "tile_flags": "on" if sparse else "off (every tile computed)", "tile_flag_density": density,
            "achieved": ach, "frac": ach / peak, "frac_vs_burst": ach / peaks["tc_burst"],
            "executed_gemm_units": units, "executed_frac": units / 4.0 * ach / peak}


def reference_formulation_gpu(B, I, T, our_ms):
    """Context for the speed claim (round-1 advisor): the REFERENCE FORMULATION of the loss - CLIP.py:34-43 written out
    with torch ops, autograd backward, fp32 with TF32 off - on the SAME B200 at the same B.  It materialises ~15 B x B
    fp32 tensors (64 GiB at B = 32768); on an allocation failure the batch is halved and the time projected (O(B^2))."""
    import torch
    import torch.nn.functional as F
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False

    def step(Bs):
        Ii = I[:Bs].detach().clone().requires_grad_(True)
        Tt = T[:Bs].detach().clone().requires_grad_(True)
        logits = (Tt @ Ii.T) / 1.0
        targets = F.softmax((Ii @ Ii.T + Tt @ Tt.T) / 2 * 1.0, dim=-1)
        tl = (-targets * F.log_softmax(logits, dim=-1)).sum(1)
        il = (-targets.T * F.log_softmax(logits.T, dim=-1)).sum(1)
        loss = ((il + tl) / 2.0).mean()
        loss.backward()
        return loss
    out = {}
    Bs = B
    while Bs >= 4096:
        try:
            step(Bs)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            l = step(Bs)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b)
            proj = ms * (B / Bs) ** 2
            out = {"ms": ms, "batch": Bs, "loss": float(l.item()), "projected_ms_at_workload_batch": proj,
                   "projected": Bs != B, "speedup_of_this_repo_device_timed": proj / our_ms,
                   "what": "torch eager fp32 (allow_tf32 = False) restatement of CLIP.py:34-43 + autograd on this GPU"}
            break
        except torch.OutOfMemoryError:
            Bs //= 2
        finally:
            torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32 = old
    return {"reference_formulation_torch_gpu_B%d" % B: out}


def single_pass_context(B, I_loc, T_loc, dev, flush, peaks, peak):
    """The same workload on the single-pass engine (`tc_f16`: fp16 operands, fp32 accumulate; stated tolerance
    5e-4 loss / 5e-3 gradients instead of the headline's fp32-class 1e-4 / 1e-3): what the sweeps reach against the
    ALGORITHMIC flop count when the logits do not have to be fp32-exact.  Context only - never the headline."""
    import torch
    ph = Phases(B, B, 0, "tc_f16", dev)
    for _ in range(3):
        ph.step(I_loc, T_loc)
    torch.cuda.synchronize()
    n, tot, phs = 5, 0.0, [0.0] * 4
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(n):
        flush.fill_(1)
        torch.cuda.synchronize()
        a.record()
        ph.step(I_loc, T_loc, record=True)
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
        for i, v in enumerate(ph.phase_ms()):
            phs[i] += v
    ms, stats_ms, bwd_ms = tot / n, phs[1] / n, phs[3] / n
    unit = 2.0 * B * B * D_EMB / 1e9   # GFLOP of one B x B x D GEMM
    return {"c4_single_pass_tc_f16_B%d" % B: {
        "ms": ms, "samples_per_s": B / (ms * 1e-3), "loss": float(ph.part.item()),
        "phases_ms": {"prepare": phs[0] / n, "stats": stats_ms, "rowloss": phs[2] / n, "bwd": bwd_ms},
        "stats_sweep_algorithmic_TFLOPs": 3 * unit / stats_ms, "stats_sweep_frac": 3 * unit / stats_ms / peak,
        "gradient_sweep_algorithmic_TFLOPs": 4 * unit / bwd_ms, "gradient_sweep_frac": 4 * unit / bwd_ms / peak,
        "gradient_sweep_frac_vs_burst": 4 * unit / bwd_ms / peaks["tc_burst"], "step_frac": 7 * unit / ms / peak, "tolerance": "loss 5e-4, gradients 5e-3 relative (tests/test_gpu_loss.py)"}}


def extras(dev, mode, peaks, peak):
    """Driver-run numbers for the other BASELINE configs (not the headline; same process, CUDA events): C2 latency (plain,
    CUDA graph, soft variant), the C5 MAE sweep corners, `cross_entropy` on materialised 8192 x 8192 inputs (plain and
    `.T` views), one ProjectionHead forward + backward per tower with its roofline terms, and the hot-path share of the
    C1 / C3 full steps.  Working sets above the 126 MB L2 are not flushed; the launch-bound ones say so."""
    import torch

    import mae_clip_b200 as m
    out = {}

    def timeit(fn, iters=20, warm=5):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    # ---- C2: loss-only microbench, B = 1024 (launch-bound: 3.8 GFLOP), default and soft variant (x 0.25, tau = 0.5)
    from mae_clip_b200.train import GraphedStep
    for tag, scale, tau in (("", 1.0, 1.0), ("_soft_x025_tau05", 0.25, 0.5)):
        I = (make_shard(1024, 0) * scale).to(dev).requires_grad_(True)
        T = (make_shard(1024, 1) * scale).to(dev).requires_grad_(True)

        def c2():
            I.grad = T.grad = None
            m.clip_contrastive_loss(I, T, tau, mode=mode).backward()
        ms = timeit(c2)
        out["c2_loss_fwd_bwd_B1024" + tag] = {"ms": ms, "samples_per_s": 1024 / (ms * 1e-3)}
        Ig, Tg = I.detach().clone().requires_grad_(True), T.detach().clone().requires_grad_(True)
        gs = GraphedStep(lambda a, b: m.clip_contrastive_loss(a, b, tau, mode=mode), [Ig, Tg], [])
        ms = timeit(lambda: gs.graph.replay())
        out["c2_loss_fwd_bwd_B1024" + tag + "_cuda_graph"] = {"ms": ms, "samples_per_s": 1024 / (ms * 1e-3)}

    # ---- C5: random masking + fused norm-pix masked MSE through the C ABI with pre-allocated outputs; algorithmic bytes of
    # SURVEY 8(d).  Corners of the sweep (N in {64, 1024} x ratio in {0.5, 0.9}) and the 0.75 centre at N = 1024
    from mae_clip_b200._lib import check as ck, cur_stream as cs, lib as L_, ptr as p_
    lib = L_()
    L, P = 196, 768

    def hbm(name, fn, nbytes, iters=10, **kw):
        ms = timeit(fn, iters=iters)
        out[name] = dict(ms=ms, GBps=nbytes / ms / 1e6, frac_hbm=nbytes / ms / 1e6 / peaks["hbm"], **kw)
        return ms

    for N, ratio in ((1024, 0.75), (1024, 0.5), (1024, 0.9), (64, 0.5), (64, 0.9)):
        keep = int(L * (1 - ratio))
        tag = "N%d_r%s" % (N, ("%g" % ratio).replace(".", ""))
        x = torch.randn(N, L, P, device=dev)
        noise = torch.rand(N, L, device=dev)
        imgs = torch.randn(N, 3, 224, 224, device=dev)
        pred = torch.randn(N, L, P, device=dev)
        dpred = torch.empty_like(pred)
        xm = torch.empty(N, keep, P, device=dev)
        mask = torch.empty(N, L, device=dev)
        restore = torch.empty(N, L, device=dev, dtype=torch.int64)
        ids_keep = torch.empty(N, keep, device=dev, dtype=torch.int64)
        loss, msum = torch.empty((), device=dev), torch.empty((), device=dev)
        ws = torch.empty(lib.mc_masked_mse_workspace_bytes(N, L), dtype=torch.uint8, device=dev)
        note = {} if N >= 512 else {"note": "working set fits L2 and the kernels are a few microseconds: launch-bound"}
        it = 10 if N >= 512 else 50
        hbm("c5_random_masking_" + tag,
            lambda: ck(lib.mc_random_masking(p_(x), 4, p_(noise), N, L, P, keep, p_(xm), p_(mask), p_(restore), p_(ids_keep), cs())),
            16 * N * L + 2 * N * keep * P * 4, iters=it, **note)
        r_eff = (L - keep) / L
        bytes_f = r_eff * N * L * P * 8 + 4 * N * L
        ms_f = hbm("c5_masked_mse_fwd_" + tag,
                   lambda: ck(lib.mc_masked_mse_fwd(p_(pred), 4, p_(imgs), p_(mask), N, 224, 224, 16, 1, p_(loss), p_(msum), p_(ws),
                                                    ws.numel(), cs())), bytes_f, iters=it, **note)
        ms_b = hbm("c5_masked_mse_bwd_" + tag,
                   lambda: ck(lib.mc_masked_mse_bwd(p_(pred), 4, p_(imgs), p_(mask), N, 224, 224, 16, 1, p_(msum), None, p_(dpred),
                                                    cs())), bytes_f + N * L * P * 4, iters=it, **note)
        out["c5_masked_mse_fwd_bwd_" + tag] = {"ms": ms_f + ms_b, "samples_per_s": N / ((ms_f + ms_b) * 1e-3)}
        del x, xm, pred, dpred, imgs

    # ---- L5: standalone cross_entropy (CLIP.py:46-52) on materialised 8192 x 8192 fp32 inputs, plain and on `.T` views
    # (CLIP.py:41); bytes: forward 2 R C 4 + 12 R, backward + 2 R C 4 (both gradients)
    R = 8192
    preds = (torch.randn(R, R, device=dev) * 4).requires_grad_(True)
    targs = torch.rand(R, R, device=dev).requires_grad_(True)
    w = torch.rand(R, device=dev)
    for tag, tr in (("", False), ("_T_views", True)):
        pv, tv = (preds.T, targs.T) if tr else (preds, targs)
        with torch.no_grad():
            hbm("cross_entropy_fwd_8192x8192" + tag, lambda: m.cross_entropy(pv, tv, reduction="none"), 2 * R * R * 4 + 12 * R)
        fwd_ms = out["cross_entropy_fwd_8192x8192" + tag]["ms"]

        def fb():
            preds.grad = targs.grad = None
            (m.cross_entropy(pv, tv, reduction="none") * w).sum().backward()
        ms = timeit(fb, iters=10)
        # the torch glue (x w, sum and their backward) moves only O(R) bytes; backward kernel = the rest of the step
        out["cross_entropy_fwd_bwd_8192x8192" + tag] = {
            "ms": ms, "bwd_ms_by_difference": ms - fwd_ms, "GBps": (6 * R * R * 4 + 12 * R) / ms / 1e6,
            "frac_hbm": (6 * R * R * 4 + 12 * R) / ms / 1e6 / peaks["hbm"]}
    del preds, targs

    # ---- L1-L2: one ProjectionHead forward + backward (dropout on), image head E = 2048 (dx needed) and text head E = 768.
    # Roofline terms: algorithmic flops of SURVEY 8(d) against the tensor peak, and the compulsory HBM bytes (x read by
    # the forward and by dW_p, dx written, 18 passes over (B, 256) fp32 tensors, the keep mask twice) against the HBM peak
    for E, need_dx in ((2048, True), (768, False)):
        Bh = 32768
        h = m.ProjectionHead(E, gemm_mode=mode).to(dev).train()
        xx = torch.randn(Bh, E, device=dev, requires_grad=need_dx)
        keepm = (torch.rand(Bh, 256, device=dev) > 0.1).to(torch.uint8)
        go = torch.randn(Bh, 256, device=dev)

        def head_step():
            for q in h.parameters():
                q.grad = None
            xx.grad = None
            h(xx, keep_mask=keepm).backward(go)
        ms = timeit(head_step, iters=10, warm=3)
        flops = 2.0 * Bh * 256 * (E + 256) * 3 - (0 if need_dx else 2.0 * Bh * E * 256)
        nbytes = Bh * E * 4.0 * (3 if need_dx else 2) + 18.0 * Bh * 256 * 4 + 2.0 * Bh * 256
        out[f"proj_head_fwd_bwd_B{Bh}_E{E}"] = {
            "ms": ms, "algorithmic_TFLOPs": flops / ms / 1e9, "samples_per_s": Bh / (ms * 1e-3),
            "roofline": {"tensor": {"achieved": flops / ms / 1e9, "peak": peak, "frac": flops / ms / 1e9 / peak,
                                    "frac_vs_burst": flops / ms / 1e9 / peaks["tc_burst"],
                                    "note": "fp32-class: every GEMM executes 3 fp16 passes, so frac <= 1/3 of the peak"},
                         "hbm": {"GBps": nbytes / ms / 1e6, "peak": peaks["hbm"], "frac": nbytes / ms / 1e6 / peaks["hbm"]},
                         "floor_ms": {"tensor_3_pass": 3 * flops / peaks["tc_burst"] / 1e9, "hbm": nbytes / peaks["hbm"] / 1e6}}}
        del h, xx, keepm, go
    torch.cuda.empty_cache()

    # ---- C1 / C3: the hot-path share of the full steps (towers are stock torch, out of scope)
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import contextlib
        import full_step_bench as fsb
        with contextlib.redirect_stdout(sys.stderr):   # stdout carries exactly one JSON line
            fsb.c1()
            torch.cuda.empty_cache()
            fsb.c3()
        out.update(fsb.out)
    except Exception as e:  # noqa: BLE001 - context numbers: never fail the bench line over a missing tower package
        out["c1_c3_full_step"] = {"unavailable": f"{type(e).__name__}: {e}"}
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
