"""Per-kernel device time of the embedding backward (sn_gather_pack_bwd) at configs[1] (B=96, T=20, V=10k, E=300), torch.profiler."""
import sys, torch
sys.path.insert(0, ".")
import icei_b200 as sn
from icei_b200 import ops
from icei_b200.packing import get_plan
import bench
from torch.profiler import profile, ProfilerActivity
dev = torch.device("cuda", 0)
B, T, V, E = 96, 20, 10000, 300
cap, lens, feat = bench.synthetic_batch(B, T, V, E, seed=0)
cap = cap.to(dev)
plan = get_plan([T] * B)
d = plan.dev(dev)
N = plan.N
dX = torch.randn(N, E, device=dev)
gE = torch.zeros(V, E, device=dev)
for p in (0.5, 0.0):
    for k in range(3):
        gE.zero_(); ops.gather_pack_bwd(cap, gE, None, True, d["row_b"], d["row_t"], None, N, dX, p, 123)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(5):
            ops.gather_pack_bwd(cap, gE, None, True, d["row_b"], d["row_t"], None, N, dX, p, 123)
        torch.cuda.synchronize()
    print("p_drop", p)
    print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12))
