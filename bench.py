#!/usr/bin/env python
"""bench.py -- decoder train tokens/sec (fwd + bwd + clamp + Adam) on the BASELINE.json config:
StyleNet FactoredLSTM, factored_size 512, emotion mode ("happy"), batch 96 per GPU, captions of length
20 over a 10k vocabulary, synthetic features (configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a kernels)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V, E, H, F, T = 10000, 300, 512, 512, 20
B_PER_GPU = 96
MODE = "happy"
METRIC = "decoder_train_tokens_per_sec"
UNIT = "tokens/s"


WORKLOAD = "factored"      # set from --workload: factored (configs[1], default) | att (configs[2]) | nic (configs[0] on GPU)
WORKLOAD_TEXT = {
    "factored": "configs[1]: StyleNet DecoderFactoredLSTM(embed 300, hidden 512, factored 512, vocab 10000), "
                "mode=happy, teacher_forcing=1.0, dropout 0.5 on, fwd+bwd+clip(0.5)+Adam, T=20",
    "att": "configs[2]: StyleNet DecoderFactoredLSTMAtt(attention 512, embed 300, hidden 512, factored 512, vocab 10000) "
           "over a 7x7x2048 feature map, mode=happy, teacher_forcing=1.0, dropout 0.5 on, "
           "CE + doubly-stochastic regulariser, fwd+bwd+clip(0.5)+Adam, T=20 (19 decoded steps)",
    "stack3": "configs[3]: 3-layer FactoredLSTM stack (embed 300, hidden 512, factored 1024, vocab 10000; 73.4 M parameters), "
              "multitask alternation: factual pass (optimizer A, lr 2e-4) / emotion pass mode=happy (optimizer B, lr 5e-4) "
              "on alternate steps, teacher_forcing=1.0, dropout 0.5 on, fwd+bwd+clip(0.5)+Adam, T=20",
    "nic": "configs[0] on the GPU: NIC DecoderRNN(embed 300, hidden 512, vocab 10000), B=64, teacher_forcing=1.0, "
           "dropout 0.5 on, fwd+bwd+clip(0.5)+Adam, T=20",
}


def workload_config(n_gpus, dtype, tokens_per_gpu=None, batch=None):
    tokens_per_gpu = tokens_per_gpu or B_PER_GPU * T
    batch = batch or B_PER_GPU
    return {
        "workload": WORKLOAD_TEXT[WORKLOAD],
        "batch_per_gpu": batch, "global_batch": batch * n_gpus, "seq_len": T,
        "tokens_per_step": tokens_per_gpu * n_gpus, "parallelism": "dp%d" % n_gpus,
        "l2": "flushed between timed steps (512 MiB write); step working set ~0.5 GB > 126 MB L2",
        "arith": dtype,
    }


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference modules on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_modules(workload):
    """(decoder class source, kind): the UNMODIFIED reference module when SN_REFERENCE_ROOT names a checkout of the
    original project, else the oracle port."""
    from oracle import port
    from oracle import reference_loader as rl
    if rl.available():
        try:
            name = {"factored": "stylenet", "stack3": "stylenet", "att": "stylenet_att", "nic": "nic"}[workload]
            return rl.load(name), "reference"
        except Exception:
            pass
    return port, "port"


def cpu_reference_run(steps, warmup, max_seconds=None, workload=None, batch=None):
    import random
    import torch
    from oracle import port
    workload = workload or WORKLOAD
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    bsz = batch or (64 if workload == "nic" else B_PER_GPU)
    mod, kind = _cpu_modules(workload)
    att = workload == "att"
    cap, lens, feats = port.synthetic_batch(bsz, T, V, E=None if att else E, feat_shape=(7, 7, 2048) if att else None,
                                            ragged=False, seed=0)
    if workload == "stack3":
        from oracle.stack import stack_forward, stack_parameters
        layers = [mod.DecoderFactoredLSTM(E if l == 0 else H, H, 1024, V, 1, dropout=0.5) for l in range(3)]
        for layer in layers:
            layer.train()
        params = stack_parameters(layers)
        opts = [torch.optim.Adam(params, lr=2e-4), torch.optim.Adam(params, lr=5e-4)]
        tgt = port.pack_targets(cap, lens)
        count = [0]

        def one_step():
            i = count[0] % 2
            count[0] += 1
            out = stack_forward(layers, cap, lens, feats, teacher_forcing_ratio=1.0, mode=("factual", MODE)[i])
            loss = torch.nn.functional.cross_entropy(out, tgt)
            for layer in layers:
                layer.zero_grad()
            loss.backward()
            port.clip_gradient(opts[i], 0.5)
            opts[i].step()
    else:
        if workload == "att":
            dec = mod.DecoderFactoredLSTMAtt(512, E, H, F, V, 1, dropout=0.5)
        elif workload == "nic":
            dec = mod.DecoderRNN(E, H, V, 1, dropout=0.5)
        else:
            dec = mod.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5)
        dec.train()
        opt = torch.optim.Adam(dec.parameters(), lr=5e-4)
        mode = None if workload == "nic" else MODE

        def one_step():
            port.train_step(dec, opt, cap, lens, feats, mode=mode, teacher_forcing_ratio=1.0, attention=att)
    random.seed(0)
    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        one_step()
        done += 1
        if max_seconds is not None and time.perf_counter() - t0 > max_seconds:
            break
    dt = time.perf_counter() - t0
    ntok = sum(lens) - (len(lens) if att else 0)
    tok = done * ntok
    return {"value": tok / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%d full steps of the same workload (B=%d, T=%d) in %.1f s, %s, torch %s CPU, %d threads"
                      % (done, bsz, T, dt, "unmodified reference module" if kind == "reference" else "oracle port",
                         torch.__version__, torch.get_num_threads()),
            "ms_per_step": 1e3 * dt / done, "steps": done}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, max(1, min(args.warmup, 2)))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, "f32 (torch CPU)"),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference arm on the host cores: the unmodified reference module when SN_REFERENCE_ROOT names a "
                "checkout of it, else oracle/port.py (its restatement, pinned at 1e-10); train step = "
                "train_multitask.py:377-389.  The reference is pure Python/torch: nothing to compile",
    }
    print(json.dumps(line), file=_JSON_OUT or sys.stdout, flush=True)


def synthetic_batch(B, Tlen, vocab, embed, seed):
    """SURVEY.md section 8d inputs: captions ~ randint(4,V), column 0 = <start>=1, last = <end>=2, fixed length
    T (N = B*T tokens), features ~ N(0,1) [B,E] (what EncoderCNN's Linear+BN emits)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    cap = torch.randint(4, vocab, (B, Tlen), generator=g)
    cap[:, 0] = 1
    cap[:, -1] = 2
    return cap, [Tlen] * B, torch.randn(B, embed, generator=g)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
_JSON_OUT = None


class ClockSampler:
    """SM clock / throttle-reason samples taken DURING the timed region.  NVML in a thread (10 ms period; a sample costs
    ~0.1 ms and no process start-up, so a 30 ms timed region at N=8 still gets samples); `nvidia-smi -lms` as the fallback
    when pynvml is missing.  The device is looked up by UUID so CUDA_VISIBLE_DEVICES remapping cannot pick another GPU."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []          # nvidia-smi text rows
        self.samples = []       # (sm, max_sm, power_w, reason_mask) from NVML
        self.proc = None
        self.nvml = None
        self.stop_flag = False
        self.source = None

    def _nvml_open(self):
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            uuid = "GPU-" + str(torch.cuda.get_device_properties(self.gpu).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        return pynvml, h

    def _nvml_loop(self):
        nv, h = self.nvml
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.samples.append((float(sm), float(mx), pw, int(mask)))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        try:
            if os.environ.get("SN_BENCH_SAMPLER", "nvml") != "nvml":
                raise RuntimeError("nvidia-smi sampler requested")
            self.nvml = self._nvml_open()
            self.source = "nvml"
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def count(self):
        return len(self.samples) if self.nvml is not None else len(self.rows)

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            nv = self.nvml[0]
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [x[0] for x in self.samples]
            mx = [x[1] for x in self.samples]
            power = [x[2] for x in self.samples if x[2] is not None]
            reasons = sorted(k for k, b in bits.items() if any(x[3] & b for x in self.samples))
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                    "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": reasons,
                    "source": "nvml, 10 ms period, during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(self.NAMES, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi -lms 50, during the timed region"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        burst = d.get("bf16_tflops", 1590.0)
        return d.get("hbm_gbs", 6650.0), (burst, d.get("bf16_tflops_sustained", burst)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, (1590.0, 1590.0), "fallback (B200_PROFILING.md)"


class Workload:
    """One training workload on this rank: model + optimizer(s) + captured step + host-side pinned inputs."""

    def __init__(self, name, precision, dev, rank, batch=None, no_graph=False, segmented=False):
        import torch
        import icei_b200 as sn
        from icei_b200 import ops
        self.name, self.precision, self.dev = name, precision, dev
        torch.manual_seed(0)                        # identical weights on every rank
        if name == "att":
            dec = sn.DecoderFactoredLSTMAtt(512, E, H, F, V, 1, dropout=0.5).to(dev)
        elif name == "nic":
            dec = sn.DecoderRNN(E, H, V, 1, dropout=0.5).to(dev)
        elif name == "stack3":
            dec = sn.DecoderFactoredLSTMStack(E, H, 1024, V, 3, dropout=0.5).to(dev)
        else:
            dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5).to(dev)
        dec.train()
        dec.set_precision(precision)
        self.dec = dec
        self.arith = "bf16 operands on tcgen05, fp32 accumulate (recurrence/softmax/Adam fp32)" if precision == "bf16" \
            else "f32 FFMA"
        opt = sn.FusedClampAdam(dec, lr=5e-4, grad_clip=0.5)
        self.trainer = sn.DataParallelTrainer(dec, opt)
        self.trainer_fac = None
        if name == "stack3":      # multitask: a second optimizer object (own Adam moments) for the factual pass
            self.trainer_fac = sn.DataParallelTrainer(dec, sn.FusedClampAdam(dec, lr=2e-4, grad_clip=0.5))
        self.bsz = bsz = batch or (64 if name == "nic" else B_PER_GPU)
        cap_h, lens, feat_h = synthetic_batch(bsz, T, V, E, seed=rank)
        self.step_kw = {"teacher_forcing_ratio": 1.0}
        if name != "nic":
            self.step_kw["mode"] = MODE
        if name == "att":
            feat_h = torch.randn(bsz, 7, 7, 2048, generator=torch.Generator().manual_seed(100 + rank))
            full_cap = cap_h
            cap_h = full_cap[:, :-1].contiguous()                  # inputs; targets = packed full[:, 1:]
            lens = [l - 1 for l in lens]
            tgt_idx = torch.cat([torch.arange(b) * T + (t + 1) for t, b in enumerate([bsz] * (T - 1))])
            self.step_kw["targets"] = full_cap.reshape(-1)[tgt_idx].to(dev)
        self.lens = lens
        self.cap_pin, self.feat_pin = cap_h.pin_memory(), feat_h.pin_memory()
        self.cap_d, self.feat_d = self.cap_pin.to(dev), self.feat_pin.to(dev)
        self.loss_pin = torch.zeros(1).pin_memory()
        self.n_tok = sum(lens)
        self.h2d = self.cap_pin.numel() * 8 + self.feat_pin.numel() * 4
        self.graphed = self.graphed_fac = None
        self.launches_per_step = None
        if not no_graph:
            # the whole step (fwd + loss + bwd [+ exchange] + clamp/Adam) captured once, replayed per step
            ops.LAUNCHES[0] = 0
            self.graphed = sn.GraphedTrainStep(self.trainer, self.cap_d, lens, self.feat_d, warmup=3,
                                               force_segmented=segmented, **self.step_kw)
            self.launches_per_step = ops.LAUNCHES[0] // 4          # 3 warm-up runs + 1 capture run
        self.kw_fac = dict(self.step_kw, mode="factual")
        if self.trainer_fac is not None and self.graphed is not None:
            self.graphed_fac = sn.GraphedTrainStep(self.trainer_fac, self.cap_d, lens, self.feat_d, warmup=3,
                                                   force_segmented=segmented, **self.kw_fac)
        self.parity = 0                                       # stack3: factual / emotion passes on alternate steps

    def _pick(self):
        if self.trainer_fac is None:
            return self.graphed, self.trainer, self.step_kw
        self.parity ^= 1
        return (self.graphed_fac, self.trainer_fac, self.kw_fac) if self.parity else (self.graphed, self.trainer, self.step_kw)

    def step_resident(self):
        g, tr, kw = self._pick()
        if g is not None:
            return g()
        return tr.step(self.cap_d, self.lens, self.feat_d, **kw)

    def step_e2e(self):
        import torch
        g, tr, kw = self._pick()
        if g is not None:
            loss, stats = g(self.cap_pin, self.feat_pin)      # pinned host -> static device buffers, then replay
        else:
            c = self.cap_pin.to(self.dev, non_blocking=True)
            f = self.feat_pin.to(self.dev, non_blocking=True)
            loss, stats = tr.step(c, self.lens, f, **kw)
        self.last = (loss, stats)
        self.loss_pin.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(self.loss_pin[0])

    def measure(self, steps, warmup, world, flush, barrier):
        """(per-step device times [ms], e2e seconds): K steps timed with CUDA events on the launching stream, L2 flushed
        between steps; then K end-to-end steps (pinned H2D + step + D2H loss + sync) on the wall clock."""
        import torch
        for _ in range(max(warmup, 3)):
            self.step_resident()
        barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.step_resident()
            e1.record()
            evs.append((e0, e1))
        barrier()
        per_step = [a.elapsed_time(b) for a, b in evs]
        for _ in range(2):
            self.step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step_e2e()
        barrier()
        return per_step, time.perf_counter() - t0


DUMP_SAMPLE = 1 << 16      # a tensor with more elements is dumped as this many elements at fixed seeded positions
DUMP_LIMIT = 64 << 20      # bytes, all files together


def dump_outputs(w, out_dir):
    """Write what the last timed step handed its caller -- the loss, the per-token stats, and the updated parameters
    with their gradients -- as DIR/<name>.npy (float32; integer stats as float64), so that two builds of the project
    can be compared output for output on the same seeded inputs."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    loss, stats = w.last
    arrays = {"loss": loss}
    arrays.update((k, v) for k, v in stats.items() if torch.is_tensor(v))
    for n, p in w.dec.named_parameters():
        arrays["param." + n] = p
        if p.grad is not None:
            arrays["grad." + n] = p.grad
    out = {}
    for name, t in arrays.items():
        t = t.detach().reshape(-1).cpu()
        if t.numel() > DUMP_SAMPLE:
            pick = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE]
            t = t[pick.sort().values]
        out[name] = t.double().numpy() if not t.is_floating_point() or t.dtype == torch.float64 else t.float().numpy()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes, more than %d" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dp_parity_check(dev, rank, world):
    """Data-parallel EQUALITY carried by the bench line (the driver's scaling run is the only place with N GPUs):
    3 steps on a fixed global batch of 12*N ragged samples through the N-GPU path (peer-fused exchange + Adam) against
    the same 3 steps on ONE GPU (computed redundantly by every rank), fp32 mode so that the only difference is the
    summation order of the gradient shards.  Reports the worst relative parameter difference and whether all ranks
    hold bit-identical parameters afterwards."""
    import torch
    import torch.distributed as dist
    import icei_b200 as sn
    from oracle import port     # synthetic_batch only (inputs); nothing of the oracle is executed on the path
    from icei_b200 import dp as _dp

    def run(precision, Vp, Ep, Hp, Fp):
        cap, lens, feats = port.synthetic_batch(12 * world, 9, Vp, E=Ep, ragged=True, seed=5)
        n_global = sum(lens)

        def make():
            torch.manual_seed(0)
            d = sn.DecoderFactoredLSTM(Ep, Hp, Fp, Vp, 1, dropout=0.0).to(dev).train().set_precision(precision)
            return d, sn.DataParallelTrainer(d, sn.FusedClampAdam(d, lr=5e-4), comm=None)
        one, _ = make()
        opt1 = sn.FusedClampAdam(one, lr=5e-4)
        loss1, lossN = [], []
        for _ in range(3):
            one.zero_grad()
            for p in one.parameters():
                p.grad = None
            l1, _ = one.forward_loss(cap.to(dev), lens, feats.to(dev), mode="happy")
            loss1.append(l1.detach().reshape(1).clone())
            opt1.step()
        dec, tr = make()
        idx, my_lens = sn.shard_lengths(lens, world, rank)
        for _ in range(3):
            lN, _ = tr.step(cap[idx].to(dev), my_lens, feats[idx].to(dev), n_global=n_global, mode="happy")
            lN = lN.detach().reshape(1).clone()
            dist.all_reduce(lN)                 # every rank holds its shard's share of the token-mean loss
            lossN.append(lN)
        torch.cuda.synchronize()
        loss_rel = max(abs(float(a) - float(b)) / max(abs(float(b)), 1e-30) for a, b in zip(lossN, loss1))
        worst = torch.zeros(1, device=dev)
        same = torch.ones(1, device=dev)
        for (n, p), (_, q) in zip(dec.named_parameters(), one.named_parameters()):
            worst = torch.maximum(worst, ((p - q).norm() / q.norm().clamp_min(1e-30)).reshape(1))
            r0 = p.detach().clone()
            dist.broadcast(r0, 0)
            if not torch.equal(r0, p.detach()):
                same.zero_()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        transport = "n/a"
        if tr.comm == "peer":
            transport = "pull (peer loads, fp32)" if _dp.PEER_FORM[0] != "push" else \
                ("push, %s gradients" % ("bf16" if tr.peers.elem_size == 2 else "fp32"))
        return {"max_rel_loss_diff_vs_1gpu": loss_rel, "max_rel_param_diff_vs_1gpu": float(worst.item()),
                "ranks_bit_identical": bool(same.item() == 1.0), "comm": tr.comm, "exchange": transport}
    r32 = run("fp32", 1000, 44, 128, 72)
    r16 = run("bf16", 1000, 40, 128, 64)
    out = dict(r32, steps=3, global_batch=12 * world,
               what="fp32 mode, ragged global batch sharded over the ranks, 3 steps vs the same steps on 1 GPU: loss of "
                    "every step (steps 2 and 3 see the updated weights) and the parameters afterwards.  The parameter "
                    "figure is dominated by elements whose summed gradient is ~0: the first Adam steps move them by "
                    "+-lr whatever the magnitude, so a last-bit difference in the sum becomes a 2*lr difference")
    out["bf16_mode"] = dict(r16, what="the same in bf16 mode (the headline's arithmetic; tolerance of the mode 2e-2): "
                                      "operand roundings are per element, the differences are accumulation order + the "
                                      "gradient transport dtype")
    return out


def decode_section(dev, cpu_seconds):
    """Greedy / beam decode throughput (BASELINE.json metric, second half) outside the headline timed region:
    greedy = forward(teacher_forcing_ratio=0) under no_grad (train_multitask.py:296-299), B=96, T=20; beam = sample()
    semantics (stylenet/model.py:198-294 with the app/backend image feed) batched over images.  Weights: reference init
    + the decode recipe of SURVEY.md section 8c.  Each figure next to the CPU port / reference on the host cores."""
    import torch
    import icei_b200 as sn
    from oracle import port
    torch.manual_seed(0)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5)
    port.sharpen_for_decode(dec)
    sd = {k: v.clone() for k, v in dec.state_dict().items()}
    dec = dec.to(dev).eval()
    g = torch.Generator().manual_seed(1)
    out = {}

    def timed(fn, reps):
        for _ in range(3):          # the 2nd call of a decode session captures its CUDA graph
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps

    B = 96
    cap = torch.randint(4, V, (B, T), generator=g)
    cap[:, 0] = 1
    feats = torch.randn(B, E, generator=g)
    cap_d, feats_d = cap.to(dev), feats.to(dev)
    for prec in ("bf16", "fp32"):
        dec.set_precision(prec)
        with torch.no_grad():
            dt = timed(lambda: dec(cap_d, [T] * B, feats_d, teacher_forcing_ratio=0.0, mode=MODE), 10)
        out["greedy_captions_per_s_" + prec] = B / dt
        for n_img in (1, 1024):
            f = torch.randn(n_img, E, generator=g).to(dev)
            dt = timed(lambda: dec.sample_batch(f, 1, 2, k=5, mode=MODE, feed_image=True), 5 if n_img == 1 else 2)
            out["beam_k5_b%d_captions_per_s_%s" % (n_img, prec)] = n_img / dt
    # CPU arm: same weights, greedy on the full batch, beam on a few images (bounded)
    mod, kind = _cpu_modules("factored")
    ref = mod.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5)
    ref.load_state_dict(sd)
    ref.eval()
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        ref(cap, [T] * B, feats, teacher_forcing_ratio=0.0, mode=MODE)
        t0 = time.perf_counter()
        n = 0
        while n < 3 and time.perf_counter() - t0 < cpu_seconds / 3:
            ref(cap, [T] * B, feats, teacher_forcing_ratio=0.0, mode=MODE)
            n += 1
        out["cpu_greedy_captions_per_s"] = B * n / (time.perf_counter() - t0)
        # beam: the image-fed variant (app/backend/model.py:386-487) exists only in the port's sample(feed_image=True)
        pref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5)
        pref.load_state_dict(sd)
        pref.eval()
        t0 = time.perf_counter()
        n = 0
        while n < 16 and time.perf_counter() - t0 < cpu_seconds / 3:
            pref.sample(feats[n:n + 1], 1, 2, k=5, mode=MODE, feed_image=True)
            n += 1
        out["cpu_beam_k5_captions_per_s"] = n / (time.perf_counter() - t0)
    out["cpu_kind"], out["cpu_cores"] = kind, os.cpu_count()
    out["note"] = "B200 figures: wall clock incl. python, features resident, ids copied back; beam_k5_b1 = one image per call"
    return out


def run_gpu(args):
    import random
    import torch
    import torch.distributed as dist
    from icei_b200 import ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    random.seed(0)
    w = Workload(WORKLOAD, args.precision, dev, rank, no_graph=args.no_graph, segmented=args.segmented,
                 batch=args.batch)
    flush = torch.empty(128 * 1024 * 1024, dtype=torch.float32, device=dev)   # 512 MiB > L2

    # ---- timed region: K steps, device time per step (CUDA events on the launching stream) -----------
    sampler = ClockSampler(local)
    sampler.start()
    ops.LAUNCHES[0] = 0
    per_step, dt_e2e = w.measure(args.steps, args.warmup, world, flush, barrier)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(w, args.dump_outputs)
    launches = ops.LAUNCHES[0] if w.graphed is None else w.launches_per_step * args.steps
    # the N-GPU == 1-GPU equality check runs AFTER the timed region (a run with it in front measured 12-15 us per step
    # more at N=2 than the same run without it: its decoders / peer mappings were still around the allocator)
    dp_parity = None
    if world > 1 and not args.no_dp_parity:
        dp_parity = dp_parity_check(dev, rank, world)
    t_local = torch.tensor([sum(per_step), dt_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
    ms_total = float(t_local[0].item())
    ms_per_step = ms_total / args.steps
    value = w.n_tok * world * args.steps / (ms_total / 1e3)
    e2e_value = w.n_tok * world * args.steps / float(t_local[1].item())

    line = None
    if rank == 0:
        hbm_peak, tf_peak, peak_src = measured_peaks()
        if args.no_roofline:
            roof, kernels = None, None
        elif WORKLOAD == "att":
            roof, kernels = att_roofline(dev, hbm_peak, peak_src)
        else:
            roof, kernels = kernel_roofline(w.dec, w.cap_d, w.lens, w.feat_d, hbm_peak, peak_src, tf_peak)
        srt = sorted(per_step)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(world, w.arith, w.n_tok, w.bsz),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": w.h2d, "d2h_bytes_per_step": 4,
                    "timing": "wall clock incl. python, pinned H2D of captions+features, D2H loss, sync per step"},
            "gpu_launches": launches, "launch_mode": "cuda-graph replay of the captured step" if w.graphed is not None
            else "eager (python-issued launches)", "clocks": clocks,
            "ms_per_step_spread": {"min": srt[0], "median": srt[len(srt) // 2], "max": srt[-1], "rank": 0},
            "roofline": roof, "kernels": kernels,
        }
        if dp_parity is not None:
            line["dp_parity"] = dp_parity
    if world > 1:
        dist.barrier()
    if rank == 0 and world == 1 and not args.no_extras:
        # ---- the rest of BASELINE.json's configs and the second half of its metric, OUTSIDE the headline region ----
        del w
        torch.cuda.empty_cache()
        cpu_s = args.cpu_seconds / 2
        extras = {}
        for name, prec in (("factored", "fp32"), ("att", "bf16"), ("stack3", "bf16"), ("nic", "bf16")):
            try:
                wx = Workload(name, prec, dev, rank)
                ps, dte = wx.measure(20, 3, 1, flush, barrier)
                r = cpu_reference_run(8, 1, max_seconds=cpu_s, workload=name)
                srt = sorted(ps)
                extras[name if prec == "bf16" else "fp32_mode"] = {
                    "workload": WORKLOAD_TEXT[name], "precision": prec, "ms_per_step": sum(ps) / len(ps),
                    "ms_per_step_spread": {"min": srt[0], "median": srt[len(srt) // 2], "max": srt[-1]},
                    "value": wx.n_tok * len(ps) / (sum(ps) / 1e3), "e2e": wx.n_tok * 20 / dte, "unit": UNIT,
                    "batch": wx.bsz, "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}}
                del wx
                torch.cuda.empty_cache()
            except Exception as exc:          # an extra must never take the headline line down
                extras[name if prec == "bf16" else "fp32_mode"] = {"error": repr(exc)[:300]}
        line["fp32_mode"] = extras.pop("fp32_mode")
        line["workloads"] = extras
        try:
            line["decode"] = decode_section(dev, args.cpu_seconds)
        except Exception as exc:
            line["decode"] = {"error": repr(exc)[:300]}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(40, 1, max_seconds=args.cpu_seconds)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), file=_JSON_OUT or sys.stdout, flush=True)
    if world > 1:
        dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the `ncu --set full` capture of the same kernels at
# B=96, T=20, H=512 (profiles/r2_a_ncu_full_k3_cluster_B96_raw.csv; the flag-synchronised kernels:
# profiles/r1_f_ncu_full_k3_bf16_B96_raw.csv); below the algorithmic bytes because W_hh is read once and most of the
# outputs are still in the 126 MB L2 when the launch ends
NCU_TRAFFIC = {"recur_fwd_cl_kernel<512>": 18.04e6 + 0.002e6, "recur_bwd_cl_kernel<512>": 26.10e6 + 0.10e6,
               "recur_fwd_bf16_kernel": 18.07e6 + 0.12e6, "recur_bwd_bf16_kernel": 26.11e6 + 0.12e6}


def att_roofline(dev, hbm_peak, peak_src):
    """K4 (attention step) timed alone at configs[2] shapes: 96 samples x 49 pixels, A=512, D=2048 (fp32 operands).
    ALGORITHMIC bytes per launch (SURVEY 8d): fwd reads att1 + features + h-side vectors, writes context + alpha;
    bwd re-reads both and read-modify-writes d att1."""
    import torch
    from icei_b200 import ops
    nb, P, A, D = 96, 49, 512, 2048
    f32 = dict(dtype=torch.float32, device=dev)
    flush = torch.empty(64 * 1024 * 1024, **f32)
    att1, feat = torch.randn(nb * P, A, **f32), torch.randn(nb, P, D, **f32)
    att2, gate_pre, wf = torch.randn(nb, A, **f32), torch.randn(nb, D, **f32), torch.randn(A, **f32)
    alpha, ctx = torch.empty(nb, P, **f32), torch.empty(nb, D, **f32)
    dctx, datt2, dgate = torch.randn(nb, D, **f32), torch.empty(nb, A, **f32), torch.empty(nb, D, **f32)
    datt1, dwf = torch.zeros(nb * P, A, **f32), torch.zeros(A, **f32)

    def timeit(fn, reps=5):
        fn()
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / reps
    t_f = timeit(lambda: ops.att_step_fwd(att1, att2, feat, wf, 0.0, gate_pre, nb, P, A, D, alpha, P, ctx, D))
    t_b = timeit(lambda: ops.att_step_bwd(att1, att2, feat, wf, 0.0, gate_pre, alpha, P, dctx, D, None, 0, nb, P, A, D,
                                          datt2, dgate, datt1, dwf, None))
    by_f = nb * (P * (A + D) * 4 + (A + D) * 4 + (D + P) * 4)
    by_b = nb * (P * (A + D) * 4 + P * A * 8 + (A + 3 * D + 2 * P) * 4)
    kernels = {"att_step_fwd_cl_kernel": {"ms": t_f, "alg_bytes": by_f, "gbs": by_f / t_f / 1e6, "frac_of_hbm_peak": by_f / t_f / 1e6 / hbm_peak},
               "att_step_bwd_cl_kernel": {"ms": t_b, "alg_bytes": by_b, "gbs": by_b / t_b / 1e6, "frac_of_hbm_peak": by_b / t_b / 1e6 / hbm_peak}}
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    roof = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["gbs"], "peak": hbm_peak, "unit": "GB/s",
            "frac": kernels[dom]["gbs"] / hbm_peak, "traffic": None, "peak_source": peak_src,
            "note": "timed alone with an L2 flush in front (the 38.5 MB fp32 feature map then comes from HBM); inside the "
                    "step the map stays in the 126 MB L2 across the 19 time steps"}
    return roof, kernels


def kernel_roofline(dec, cap_d, lens, feat_d, hbm_peak, peak_src, tf_peak=(1638.2, 1368.6)):
    """Per-kernel device time (CUDA events, L2 flushed) of the HBM-bound kernels of one step, the roofline
    object for the dominant one, and a large-batch point of the same kernel (B=4096/GPU) where the serial
    chain no longer hides the memory system.  ALGORITHMIC bytes per launch as defined in DESIGN.md."""
    import torch
    import icei_b200 as sn
    from icei_b200 import ops
    dev = cap_d.device
    f32 = dict(dtype=torch.float32, device=dev)
    b16 = dict(dtype=torch.bfloat16, device=dev)
    flush = torch.empty(64 * 1024 * 1024, **f32)
    bf16 = dec.bf16
    Whh, bhh = dec._recurrent_weights()
    Wb = Whh.bfloat16().contiguous()

    def timeit(fn, reps=5):
        fn()
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / reps

    def recur_pair(lengths):
        plan = sn.get_plan(lengths)
        d = plan.dev(dev)
        N, B, TT = plan.N, plan.B, plan.T
        XP = torch.randn(N, 4 * H, **f32)
        Hall, Call = torch.empty(N, H, **f32), torch.empty(N, H, **f32)
        gates = torch.empty(N, 4 * H, **f32)
        dH = torch.randn(N, H, **f32)
        dZ = torch.empty(N, 4 * H, **f32)
        if bf16 and B >= ops.RECUR_GEMM_MIN_BATCH[0]:
            # what the decoder runs at this batch size: one tcgen05 GEMM per step, cell fused into the epilogue
            Hb, dZb = torch.empty(N, H, **b16), torch.empty(N, 4 * H, **b16)
            Wil = ops.cast_gate_interleave(Whh)
            dcar = torch.empty(B, H, **f32)

            def fwd():
                ops.recur_fwd_gemm(dec.cell, H, B, plan, XP, Wil, bhh, Hall, Hb, Call, gates)

            def bwd():
                ops.recur_bwd_gemm(dec.cell, H, B, plan, Wb, Call, gates, dH, dZ, dZb, dcar)
            fwd(); bwd()
            torch.cuda.synchronize()
            graphs = []
            for fn in (fwd, bwd):          # replayed from a CUDA graph, like the training step
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph):
                    fn()
                graphs.append(gph)
            fwd, bwd = graphs[0].replay, graphs[1].replay
            by_f = N * H * (16 + 8 + 16 + 4 + 4) + 4 * H * H * 2
            by_b = N * H * (16 + 16 + 8 + 4 + 8 + 8) + 4 * H * H * 2
            names = ("recur_fwd_gemm(cell epilogue) x%d steps" % TT, "recur_bwd_gemm(cell epilogue) x%d steps" % TT)
        elif bf16:
            Hb, Hpb, dZb = torch.empty(N, H, **b16), torch.empty(N, H, **b16), torch.empty(N, 4 * H, **b16)

            def fwd():
                cst = torch.zeros(B, H, **f32)
                ops.recur_fwd_bf16(dec.cell, H, B, d["bs"], d["off"], 0, TT, XP, Wb, bhh, None, Hall, Hb, Hpb, Call,
                                   gates, cst)

            def bwd():
                dh, dc = torch.zeros(B, H, **f32), torch.zeros(B, H, **f32)
                ops.recur_bwd_bf16(dec.cell, H, B, d["bs"], d["off"], 0, TT, Wb, None, Call, gates, dH, dZ, dZb, dh, dc)
            # XP + c in/out + gates + h fp32 + h bf16 x2 ; W_hh bf16 once
            by_f = N * H * (16 + 8 + 16 + 4 + 4) + 4 * H * H * 2
            by_b = N * H * (16 + 16 + 8 + 4 + 8 + 8) + 4 * H * H * 2
            names = ("recur_fwd_cl_kernel<%d>" % H, "recur_bwd_cl_kernel<%d>" % H) if ops.recur_cluster_ok(H, B) \
                else ("recur_fwd_bf16_kernel", "recur_bwd_bf16_kernel")
        else:
            Hprev = torch.empty(N, H, **f32)

            def fwd():
                cst = torch.zeros(B, H, **f32)
                ops.recur_fwd(dec.cell, H, B, d["bs"], d["off"], 0, TT, XP, Whh, bhh, None, Hall, Call, Hprev, gates, cst)

            def bwd():
                dh, dc = torch.zeros(B, H, **f32), torch.zeros(B, H, **f32)
                ops.recur_bwd(dec.cell, H, B, d["bs"], d["off"], 0, TT, Whh, None, Call, gates, dH, dZ, dh, dc)
            by_f = N * H * 48 + 4 * H * H * 4
            by_b = N * H * 52 + 4 * H * H * 4
            names = ("recur_fwd_kernel", "recur_bwd_kernel")
        t_f, t_b = timeit(fwd), timeit(bwd)
        return {names[0]: {"ms": t_f, "alg_bytes": by_f, "gbs": by_f / t_f / 1e6},
                names[1]: {"ms": t_b, "alg_bytes": by_b, "gbs": by_b / t_b / 1e6}}

    kernels = recur_pair(lens)
    N = sum(lens)
    logits = torch.randn(N, V, **f32)
    tgt = torch.randint(0, V, (N,), device=dev)
    rl = torch.empty(N, **f32)

    def smx():
        ops.softmax_nll(logits, N, V, targets=tgt, row_loss=rl, dlogits=logits, grad_scale=1.0 / N)

    t_s = timeit(smx)
    kernels["softmax_nll_kernel"] = {"ms": t_s, "alg_bytes": N * V * 8, "gbs": N * V * 8 / t_s / 1e6}
    a = dec.arena()
    npar = a.total
    m_, v_ = torch.zeros_like(a.flat), torch.zeros_like(a.flat)
    pcopy, gcopy = a.flat.clone(), torch.randn_like(a.flat) * 0.01

    def adam():
        ops.adam_clamp(pcopy, gcopy, m_, v_, [(0, npar)], [1e-3], [0.1], 0.9, 0.999, 1e-8, 0.5)

    t_a = timeit(adam)
    kernels["adam_clamp_kernel"] = {"ms": t_a, "alg_bytes": npar * 28, "gbs": npar * 28 / t_a / 1e6}
    del logits, m_, v_, pcopy, gcopy
    big = recur_pair([T] * 4096)
    huge = recur_pair([T] * 16384) if bf16 else None
    dom = max((k for k in kernels if k.startswith("recur")), key=lambda k: kernels[k]["ms"])
    ach = kernels[dom]["gbs"]
    bigdom = max(big, key=lambda k: big[k]["ms"])
    roof = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
            "frac": ach / hbm_peak, "traffic": NCU_TRAFFIC.get(dom) if len(lens) == 96 else None,
            "traffic_source": "ncu --set full, profiles/r2_a_ncu_full_k3_cluster_B96_raw.csv", "peak_source": peak_src,
            "note": "latency-bound at B=96: T serial steps, each with an exchange of h_t between the 16 CTAs of a cluster "
                    "through distributed shared memory (DESIGN.md 4). "
                    "At B=4096/GPU the recurrence runs as per-step tcgen05 GEMMs with the cell in the epilogue "
                    "(throughput regime): %.0f GB/s = %.2f of peak" % (big[bigdom]["gbs"], big[bigdom]["gbs"] / hbm_peak),
            "large_batch": {"B": 4096, "kernel": bigdom, "achieved": big[bigdom]["gbs"],
                            "frac": big[bigdom]["gbs"] / hbm_peak}}
    kernels["large_batch_B4096"] = big
    if huge:
        kernels["large_batch_B16384"] = huge
        for k in huge:
            huge[k]["frac_of_hbm_peak"] = huge[k]["gbs"] / hbm_peak
    for k in big:
        big[k]["frac_of_hbm_peak"] = big[k]["gbs"] / hbm_peak
    if bf16:
        kernels["tensor"] = gemm_tensor_points(timeit, dev, tf_peak)
    return roof, kernels


def gemm_tensor_points(timeit, dev, tf_peak):
    """Tensor-pipe side of the path: the CTA-pair tcgen05 GEMM (sn_gemm2.cu) on the projection / vocabulary shapes of
    configs[1] at B=96 (N=1920 tokens: latency regime) and at B=4096 (N=81920: throughput regime).  TFLOP/s on
    2*M*N*K and the fraction of the MEASURED cuBLAS bf16 peaks (burst: a kernel timed alone; sustained: back to back for
    seconds, power-limited); ncu sm__pipe_tensor_cycles_active of the same kernels:
    profiles/r1_i_ncu_full_gemm_pair_N40960_raw.csv."""
    import torch
    from icei_b200 import ops
    out = {"peak_tflops_burst": tf_peak[0], "peak_tflops_sustained": tf_peak[1]}
    b16 = dict(dtype=torch.bfloat16, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)

    def point(t, fl):
        tf = fl / t / 1e9
        return {"ms": t, "tflops": tf, "frac_of_burst_peak": tf / tf_peak[0], "frac_of_sustained_peak": tf / tf_peak[1]}

    for ntok in (T * B_PER_GPU, T * 4096):
        tag = "N%d" % ntok
        X = torch.randn(ntok, 304, **b16)
        Vw = torch.randn(4 * F, 304, **b16)
        A1 = torch.empty(ntok, 4 * F, **b16)
        t = timeit(lambda: ops.gemm_bf16(ops.OP_NT, X, Vw, ntok, 4 * F, 304, 304, 304, Cb=A1, ldcb=4 * F, impl="pair"))
        fl = 2.0 * ntok * 4 * F * 304
        out["V_stage_" + tag] = point(t, fl)
        Hb = torch.randn(ntok, H, **b16)
        Cw = (torch.randn(V, H, **f32) / 8).bfloat16()
        bias = torch.zeros(V, **f32)
        tgt = torch.randint(0, V, (ntok,), device=dev)
        tl, lse, rl = torch.empty(ntok, **f32), torch.empty(ntok, **f32), torch.empty(ntok, **f32)
        am = torch.empty(ntok, dtype=torch.int64, device=dev)
        ab = torch.zeros(ntok, dtype=torch.int32, device=dev)
        dLb = torch.empty(ntok, V, **b16)
        fl = 2.0 * ntok * V * H
        t = timeit(lambda: ops.vocab_nll_fwd(Hb, Cw, bias, tgt, ntok, V, H, tl, lse, rl, am, ab))
        out["vocab_nll_fwd_" + tag] = dict(point(t, fl), hbm_bytes_logits=0)
        t = timeit(lambda: ops.vocab_nll_bwd(Hb, Cw, bias, tgt, ntok, V, H, tl, lse, 1.0 / ntok, dLb, ab, None))
        out["vocab_nll_bwd_" + tag] = point(t, fl)
        dH = torch.empty(ntok, H, **f32)
        t = timeit(lambda: ops.gemm_bf16(ops.OP_NN, dLb, Cw, ntok, H, V, V, H, C=dH, ldc=H, impl="pair"))
        out["vocab_dH_" + tag] = point(t, fl)
        del X, A1, Hb, dLb, dH
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every launch from python instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--workload", default="factored", choices=["factored", "att", "nic", "stack3"])
    ap.add_argument("--batch", type=int, default=None,
                    help="samples per GPU (default: the BASELINE config, 96; e.g. 4096 = throughput regime, a supplementary point)")
    ap.add_argument("--no-roofline", action="store_true", help="skip the per-kernel roofline section (launch lists of the step only)")
    ap.add_argument("--segmented", action="store_true", help="force the 3-graph (data-parallel) replay form on one GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the fp32-mode / other-config / decode sections of the line")
    ap.add_argument("--no-dp-parity", action="store_true", help="skip the N-GPU == 1-GPU equality check (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, stats, parameters, gradients; "
                         "large tensors as a fixed seeded sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    global WORKLOAD, B_PER_GPU
    WORKLOAD = args.workload
    if args.batch:
        B_PER_GPU = args.batch
    # stdout carries the ONE JSON line and nothing else: libraries that write to fd 1 (NCCL's version banner, a
    # compiler note from a child process) are sent to stderr while the run is in progress
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
