#!/usr/bin/env python
"""ROUGE-L on the GPU (``icei_b200.rouge``, kernel K13) against the CPU restatement of coco-caption's scorer
(``oracle/rouge.py``) and, when it is importable, pycocoevalcap itself, on one GPU.

    python bench_rouge.py [--sizes 1000,5000] [--refs 5] [--repeat 20] [--launches 200] [--out PATH]

Corpora are bench_cider.py's: seeded and shaped like captions (per image a "scene" of 24 ids from a 10 000-word
vocabulary; the hypothesis and its references are random spans of it of 8..20 ids with 20 % of the ids replaced).
Per corpus size it reports:
  e2e_ms       corpus_rouge(refs, hyps) end to end -- checks, packing, the host-to-device copy, the kernel, the copy back
               and the mean (the call returns numpy data, so it ends synchronised); median over --repeat calls
  reuse_ms     RougeL(refs).compute_score(hyps) on a RougeL made once: hypotheses packed and scored (median)
  pack_ms      the host-side packing alone (median)
  kernel_ms    sn_rouge_l alone: CUDA events around --launches launches
  rows_ms      RougeL.score_samples at the self-critical training shape: 96 images x 5 samples, seqs [480, 42]
               (max_seq_length 40) with every row at its full length; median over --repeat synchronised calls
  oracle_ms    the CPU restatement on this host (one call)
  coco_ms      pycocoevalcap's Rouge().compute_score on the ids joined as words (null when absent)
  agree        GPU per-image scores bitwise equal to the oracle's (and to pycocoevalcap's when present), RougeL equal to
               corpus_rouge, and the rows form with identity ids equal to compute_score
One JSON line, with the device name and power limit read in the same run and, per corpus, the SM clock sampled during
its timed calls (bench.py's ClockSampler); also written to --out."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SCST_IMAGES, SCST_SAMPLES, SCST_WIDTH = 96, 5, 42


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,5000")
    ap.add_argument("--refs", type=int, default=5)
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rouge_bench_N1.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_rouge.py needs a CUDA device (there is no CPU path to measure)")
    from bench import ClockSampler
    from bench_cider import VOCAB, corpus, device_info, event_ms
    from icei_b200 import bleu, ops, rouge
    from oracle import rouge as oracle_rouge
    try:
        from pycocoevalcap.rouge.rouge import Rouge
    except ImportError:
        Rouge = None
    info = device_info()
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = []
    for i, n in enumerate(int(s) for s in args.sizes.split(",")):
        refs, hyps = corpus(n, args.refs, seed=2000 + i)
        tokens = sum(map(len, hyps)) + sum(len(r) for rs in refs for r in rs)

        def timed(fn):
            for _ in range(3):
                fn()
            ms = []
            for _ in range(args.repeat):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = fn()
                torch.cuda.synchronize()
                ms.append(1e3 * (time.perf_counter() - t0))
            return out, ms
        clocks = ClockSampler(torch.cuda.current_device())
        clocks.start()
        (mean, got), e2e = timed(lambda: rouge.corpus_rouge(refs, hyps))
        scorer = rouge.RougeL(refs)
        (mean_r, got_r), reuse = timed(lambda: scorer.compute_score(hyps))
        pack = []
        for _ in range(args.repeat):
            t0 = time.perf_counter()
            bleu._pack(refs, hyps)
            pack.append(1e3 * (time.perf_counter() - t0))
        # the kernel alone, on the packed device corpus
        views, max_len = rouge._upload(refs, hyps)
        out = torch.empty(n, dtype=torch.float64, device=dev)
        kernel_ms = event_ms(lambda: ops.rouge_l(*views, max_len, rouge.BETA2, out=out), args.launches)
        # self-critical rewards: random full-length rows against random images of the corpus
        g = torch.Generator().manual_seed(3000 + i)
        R = SCST_IMAGES * SCST_SAMPLES
        seqs = torch.randint(3, VOCAB, (R, SCST_WIDTH), generator=g)
        seqs[:, 0] = 1
        seqs = seqs.to(dev)
        lengths = torch.full((R,), SCST_WIDTH, dtype=torch.int64, device=dev)
        ids = np.repeat(torch.randint(0, n, (SCST_IMAGES,), generator=g).numpy(), SCST_SAMPLES)
        _, rows_t = timed(lambda: scorer.score_samples(seqs, lengths, ids, 1, 2))
        clocks = clocks.stop()
        ident = scorer.score_samples(seqs[:min(n, R)], lengths[:min(n, R)], np.arange(min(n, R)), 1, 2).cpu().numpy()
        hyps_ident = [s[1:] for s in seqs[:min(n, R)].cpu().tolist()] + hyps[R:]
        t0 = time.perf_counter()
        want_mean, want = oracle_rouge.corpus_rouge(refs, hyps)
        oracle_ms = 1e3 * (time.perf_counter() - t0)
        ok = (np.array_equal(got, want) and mean == want_mean and mean_r == mean and np.array_equal(got_r, got)
              and np.array_equal(ident, scorer.compute_score(hyps_ident)[1][:min(n, R)]))
        coco_ms = None
        if Rouge is not None:
            gts = {j: [" ".join(map(str, r)) for r in rs] for j, rs in enumerate(refs)}
            res = {j: [" ".join(map(str, h))] for j, h in enumerate(hyps)}
            t0 = time.perf_counter()
            _, coco = Rouge().compute_score(gts, res)
            coco_ms = 1e3 * (time.perf_counter() - t0)
            ok = ok and np.array_equal(np.asarray(coco), got)
        rows.append({"n_img": n, "refs_per_img": args.refs, "tokens": tokens,
                     "e2e_ms": round(statistics.median(e2e), 3), "e2e_ms_min": round(min(e2e), 3),
                     "reuse_ms": round(statistics.median(reuse), 3), "pack_ms": round(statistics.median(pack), 3),
                     "kernel_ms": round(kernel_ms, 4), "rows_ms": round(statistics.median(rows_t), 3),
                     "rows_shape": [R, SCST_WIDTH], "oracle_ms": round(oracle_ms, 1),
                     "coco_ms": None if coco_ms is None else round(coco_ms, 1), "agree": ok, "rouge_l": mean,
                     "sm_clock_mhz": clocks.get("sm_mhz"), "sm_clock_max_mhz": clocks.get("sm_max_mhz"),
                     "clock_reasons": clocks.get("reasons")})
    line = json.dumps(dict({"bench": "ROUGE-L (beta=1.2)"}, **info, corpora=rows))
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
