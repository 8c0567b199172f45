"""Kernel timeline of one CUDA-graph replay of the configs[1] training step (torch.profiler / CUPTI)."""
import sys, json, random, torch
sys.path.insert(0, ".")
import icei_b200 as sn
from torch.profiler import profile, ProfilerActivity
import bench
E, H, F, V, T, B = 300, 512, 512, 10000, 20, 96
torch.manual_seed(0)
dev = torch.device("cuda", 0)
dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5).to(dev); dec.train(); dec.set_precision("bf16")
opt = sn.FusedClampAdam(dec, lr=5e-4, grad_clip=0.5)
tr = sn.DataParallelTrainer(dec, opt)
cap, lens, feat = bench.synthetic_batch(B, T, V, E, seed=0)
cap, feat = cap.to(dev), feat.to(dev)
random.seed(0)
g = sn.GraphedTrainStep(tr, cap, lens, feat, warmup=3, teacher_forcing_ratio=1.0, mode="happy")
for _ in range(5): g()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
    for _ in range(3):
        g()
    torch.cuda.synchronize()
ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name and "Memset" not in e.name]
ev.sort(key=lambda e: e.time_range.start)
# split into replays by large gaps
# (measured from the latest END so far: a short kernel that starts under a long one on another stream is no gap)
groups, cur = [], [ev[0]]
last_end = ev[0].time_range.end
for b in ev[1:]:
    if b.time_range.start - last_end > 100:  # us
        groups.append(cur); cur = []
    cur.append(b)
    last_end = max(last_end, b.time_range.end)
groups.append(cur)
rep = groups[-1]
t0 = rep[0].time_range.start
end = max(e.time_range.end for e in rep)
print("replay: %d kernels, span %.1f us" % (len(rep), end - t0))
busy = 0.0; last = t0
for e in rep:
    s, f = e.time_range.start, e.time_range.end
    if f > last:
        busy += f - max(s, last); last = f
print("union busy %.1f us, idle %.1f us" % (busy, end - t0 - busy))
for e in rep:
    print("%8.1f %7.1f  %s" % (e.time_range.start - t0, e.time_range.end - e.time_range.start, e.name[:90]))
