#!/usr/bin/env python
"""Corpus BLEU-1..4 on the GPU (``icei_b200.bleu.corpus_bleu``, kernel K10) against the CPU restatement of nltk's
corpus_bleu (``oracle/bleu.py``) and, when it is importable, nltk itself, on one GPU.

    python bench_bleu.py [--sizes 1000,5000] [--refs 5] [--repeat 20] [--launches 200]

Corpora are seeded: per item a "scene" of 42 ids from a 10 000-word vocabulary, and the hypothesis and its references
are random spans of it (lengths 0..42) with 20 % of the ids replaced, so every n-gram order has matches.  Per corpus
size it reports:
  e2e_ms     corpus_bleu(refs, hyps, [BLEU-1..4 weights]) end to end -- packing, the host-to-device copy, the kernel,
             the column sum and the 10-integer copy back (the call returns Python floats, so it ends synchronised);
             median over --repeat calls after warm-up
  pack_ms    the host-side packing alone (median)
  kernel_ms  the kernel alone: CUDA events around --launches launches on the packed corpus, per launch
  oracle_ms  the CPU restatement on this host (one call for the four weight tuples)
  nltk_ms    nltk's corpus_bleu, once per weight tuple as the reference calls it (null when nltk is absent)
  equal      GPU scores == oracle scores, all four, exactly
One JSON line, with the device name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
W4 = [(1.0,), (0.5, 0.5), (1 / 3, 1 / 3, 1 / 3), (0.25, 0.25, 0.25, 0.25)]
VOCAB, MAX_LEN = 10000, 42


def corpus(n, n_refs, seed):
    import numpy as np
    rng = np.random.default_rng(seed)

    def spans(scene, k):
        L = rng.integers(0, MAX_LEN + 1, k)
        s0 = rng.integers(0, MAX_LEN - L + 1)
        out = []
        for l, s in zip(L.tolist(), s0.tolist()):
            x = scene[s:s + l].copy()
            sub = rng.random(l) < 0.2
            x[sub] = rng.integers(0, VOCAB, int(sub.sum()))
            out.append(x.tolist())
        return out
    refs, hyps = [], []
    for _ in range(n):
        scene = rng.integers(0, VOCAB, MAX_LEN)
        sents = spans(scene, n_refs + 1)
        hyps.append(sents[0])
        refs.append(sents[1:])
    return refs, hyps


def device_info():
    import torch
    name = torch.cuda.get_device_name(torch.cuda.current_device())
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        power = float(out.stdout.strip().splitlines()[0])
    except Exception:       # the number is reported as unknown rather than guessed
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,5000")
    ap.add_argument("--refs", type=int, default=5)
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_bleu.py needs a CUDA device (there is no CPU path to measure)")
    import icei_b200 as sn
    from icei_b200 import bleu
    from oracle import bleu as oracle_bleu
    try:
        from nltk.translate import bleu_score as nltk_bleu
    except ImportError:
        nltk_bleu = None
    name, power = device_info()
    rows = []
    for i, n in enumerate(int(s) for s in args.sizes.split(",")):
        refs, hyps = corpus(n, args.refs, seed=1000 + i)
        tokens = sum(map(len, hyps)) + sum(len(r) for rs in refs for r in rs)
        for _ in range(3):
            got = bleu.corpus_bleu(refs, hyps, W4)
        e2e = []
        for _ in range(args.repeat):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = bleu.corpus_bleu(refs, hyps, W4)
            torch.cuda.synchronize()
            e2e.append(1e3 * (time.perf_counter() - t0))
        pack = []
        for _ in range(args.repeat):
            t0 = time.perf_counter()
            bleu._pack(refs, hyps)
            pack.append(1e3 * (time.perf_counter() - t0))
        # the kernel alone, on the packed device buffer
        buf, (nh, R, Th, Tr), max_len, max_group = bleu._pack(refs, hyps)
        dev = torch.from_numpy(buf).cuda()
        k = 2 * nh + R + 3
        tok = dev[k:].view(torch.int32)
        a = (tok[:Th], dev[:nh + 1], tok[Th:Th + Tr], dev[nh + 1:nh + R + 2], dev[nh + R + 2:k], max_len, max_group)
        for _ in range(10):
            sn.ops.bleu_counts(*a)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.launches):
            sn.ops.bleu_counts(*a)
        ev1.record()
        ev1.synchronize()
        kernel_ms = ev0.elapsed_time(ev1) / args.launches
        t0 = time.perf_counter()
        want = oracle_bleu.corpus_bleu(refs, hyps, W4)
        oracle_ms = 1e3 * (time.perf_counter() - t0)
        nltk_ms = None
        if nltk_bleu is not None:
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                t0 = time.perf_counter()
                for w in W4:
                    nltk_bleu.corpus_bleu(refs, hyps, w)
                nltk_ms = 1e3 * (time.perf_counter() - t0)
        rows.append({"n_hyp": n, "refs_per_hyp": args.refs, "tokens": tokens,
                     "e2e_ms": round(statistics.median(e2e), 3), "e2e_ms_min": round(min(e2e), 3),
                     "pack_ms": round(statistics.median(pack), 3), "kernel_ms": round(kernel_ms, 4),
                     "oracle_ms": round(oracle_ms, 1), "nltk_ms": None if nltk_ms is None else round(nltk_ms, 1),
                     "equal": got == want, "bleu": got})
    print(json.dumps({"bench": "corpus_bleu BLEU-1..4", "device": name, "power_limit_w": power,
                      "corpora": rows}))


if __name__ == "__main__":
    main()
