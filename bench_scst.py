#!/usr/bin/env python
"""One self-critical training step (``icei_b200.scst.scst_step``) of the configs[1] model on one GPU.

    python bench_scst.py [--images 96] [--n 5] [--precision bf16] [--repeat 20] [--no-cpu-oracle] [--out PATH]

Model: DecoderFactoredLSTM(embed 300, hidden 512, factored 512, vocab 10 000), max_seq_length 40, reference init
(flat logits, so most samples run to the length limit: the longest sampling decode).  Rewards are scored against a
seeded caption-like corpus of 1 000 training images x 5 references (bench_cider.corpus); the step's images are the
first --images of it.  Device time per phase, median over --repeat, each phase bracketed by CUDA events and ending in
a synchronise:
  sample_ms   sample_captions: n samples per image (K12)
  greedy_ms   sample_captions(greedy=True): the greedy baseline
  reward_ms   CiderD.score_samples of the samples and of the greedy captions (K11)
  train_ms    advantages, the length sort (one device-to-host copy), token weights, forward_loss with token_weights
              (forward + backward) and the fused clamp + Adam
  total_ms    scst_step(baseline="greedy") end to end
  cpu_oracle_ms  oracle/scst.py's reference step on this host's CPU (one call, given the GPU's samples), for context
One JSON line with the device name and power limit read in the same run; also written to --out."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def timed(fn, repeat):
    import torch
    times = []
    for _ in range(repeat):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=96)
    ap.add_argument("--n", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--no-cpu-oracle", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import icei_b200 as sn
    from icei_b200.packing import get_plan
    from bench_cider import corpus, device_info
    if not torch.cuda.is_available():
        raise SystemExit("bench_scst.py measures the GPU: no CUDA device")
    START, END = 1, 2
    E, H, F, V = 300, 512, 512, 10000
    torch.manual_seed(0)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.22).cuda().set_precision(args.precision)
    dec.train()
    opt = sn.FusedClampAdam(dec, lr=5e-5, grad_clip=0.5)
    refs, _ = corpus(1000, 5, 0)
    cd = sn.cider.CiderD(refs)
    B, n = args.images, args.n
    ids = list(range(B))
    feats = torch.randn(B, E, generator=torch.Generator().manual_seed(1)).cuda()
    state = {}

    def sample():
        state["s"] = dec.sample_captions(feats, START, END, n=n, seed=3)

    def greedy():
        state["g"] = dec.sample_captions(feats, START, END, n=1, greedy=True)

    def reward():
        s, g = state["s"], state["g"]
        state["r"] = cd.score_samples(s[0], s[1], np.repeat(ids, n), START, END)
        state["rg"] = cd.score_samples(g[0], g[1], ids, START, END)

    def train():
        seqs, lens, _ = state["s"]
        adv, _ = sn.scst.advantages(state["r"], n, "greedy", state["rg"])
        lens_h = lens.cpu().tolist()
        order = sn.scst.sort_by_length(lens_h)
        idx = torch.tensor(order, dtype=torch.int64).cuda()
        lens_s = [lens_h[r] for r in order]
        w = sn.scst.token_weights(adv.index_select(0, idx), get_plan(lens_s))
        opt.zero_grad()
        dec.forward_loss(seqs.index_select(0, idx), lens_s, feats.index_select(0, idx // n), token_weights=w,
                         n_global=sum(lens_s) - len(lens_s))
        opt.step()

    it = [0]

    def total():
        it[0] += 1
        sn.scst.scst_step(dec, opt, cd, feats, ids, START, END, n=n, baseline="greedy", seed=it[0])

    for fn in (sample, greedy, reward, train, total):       # warm-up: sessions, graphs, plans, allocator
        fn()
        fn()
    res = {"bench": "scst_step", "model": "configs[1] DecoderFactoredLSTM(300, 512, 512, 10000)",
           "precision": args.precision, "images": B, "samples_per_image": n, "max_seq_length": dec.max_seq_length,
           "corpus_images": len(refs)}
    res.update(device_info())
    for name, fn in (("sample_ms", sample), ("greedy_ms", greedy), ("reward_ms", reward), ("train_ms", train),
                     ("total_ms", total)):
        res[name] = round(timed(fn, args.repeat), 3)
    lens = state["s"][1]
    res["mean_sample_length"] = round(float(lens.double().mean()), 2)
    res["sampled_tokens"] = int((lens - 1).sum())
    if not args.no_cpu_oracle:
        from oracle import port, scst as so
        ref = port.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.0)
        ref.load_state_dict({k: v.cpu() for k, v in dec.state_dict().items()})
        ropt = torch.optim.Adam(ref.parameters(), lr=5e-5)
        seqs, lens, _ = state["s"]
        g = state["g"]
        t0 = time.perf_counter()
        so.reference_step(lambda c, l, f: ref(c, l, f, teacher_forcing_ratio=1.0), list(ref.parameters()), ropt, refs,
                          feats.cpu(), ids, seqs.cpu(), lens.cpu(), n, "greedy", END, g[0].cpu(), g[1].cpu())
        res["cpu_oracle_ms"] = round(1000 * (time.perf_counter() - t0), 1)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
