"""Per-rank work of the 8-GPU job on ONE GPU: the three sweeps over a 4096-row strip of B = 32768 (tools only)."""
import sys, json
sys.path.insert(0, ".")
import torch
import bench
B, b = 32768, int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda")
I = torch.cat([bench.make_shard(4096, 1000 + k) for k in range(8)]).to(dev)
T = torch.cat([bench.make_shard(4096, 5000 + k) for k in range(8)]).to(dev)
ph = bench.Phases(B, b, 0, "tc_f16x3", dev)
for _ in range(3): ph.step(I, T)
torch.cuda.synchronize()
acc = [0.0] * 4
n = 10
for _ in range(n):
    ph.step(I, T, record=True)
    torch.cuda.synchronize()
    for i, v in enumerate(ph.phase_ms()): acc[i] += v
print("prepare %.3f stats %.3f rowloss %.3f bwd %.3f" % tuple(a / n for a in acc))
