#!/usr/bin/env python
"""CIDEr-D on the GPU (``icei_b200.cider``, kernels K11) against the CPU restatement of coco-caption's scorer
(``oracle/cider.py``) and, when it is importable, pycocoevalcap itself, on one GPU.

    python bench_cider.py [--sizes 1000,5000] [--refs 5] [--repeat 20] [--launches 200] [--out PATH]

Corpora are seeded and shaped like captions: per image a "scene" of 24 ids from a 10 000-word vocabulary, and the
hypothesis and its references are random spans of it of 8..20 ids with 20 % of the ids replaced, so every n-gram order
has matches and document frequencies vary.  Per corpus size it reports:
  e2e_ms       corpus_cider(refs, hyps) end to end -- checks, packing, the host-to-device copy, both kernels, the copy
               back and the mean (the call returns numpy data, so it ends synchronised); median over --repeat calls
  ciderd_ms    CiderD(refs).compute_score(hyps) on a CiderD made once: hypotheses packed and scored (median)
  pack_ms      the host-side packing alone (median)
  df_ms        sn_cider_df alone (clearing the table, then counting): CUDA events around --launches launches
  scores_ms    sn_cider_scores alone, the same way
  oracle_ms    the CPU restatement on this host (one call)
  coco_ms      pycocoevalcap's Cider(n=4, sigma=6.0).compute_score on the ids joined as words (null when absent)
  agree        GPU per-image scores within 1e-12 * max(1, |x|) of the oracle's (and of pycocoevalcap's when present)
One JSON line, with the device name and power limit read in the same run and, per corpus, the SM clock sampled during
its timed calls (bench.py's ClockSampler); also written to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
VOCAB, SCENE, MIN_LEN, MAX_LEN = 10000, 24, 8, 20


def corpus(n, n_refs, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    refs, hyps = [], []
    for _ in range(n):
        scene = rng.integers(0, VOCAB, SCENE)
        sents = []
        for L in rng.integers(MIN_LEN, MAX_LEN + 1, n_refs + 1).tolist():
            s0 = int(rng.integers(0, SCENE - L + 1))
            x = scene[s0:s0 + L].copy()
            sub = rng.random(L) < 0.2
            x[sub] = rng.integers(0, VOCAB, int(sub.sum()))
            sents.append(x.tolist())
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
    return {"device": name, "power_limit_w": power}


def agree(got, want):
    import numpy as np
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return bool(np.all(np.abs(got - want) <= 1e-12 * np.maximum(1.0, np.abs(want))))


def event_ms(fn, launches):
    import torch
    for _ in range(10):
        fn()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(launches):
        fn()
    ev1.record()
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,5000")
    ap.add_argument("--refs", type=int, default=5)
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cider_bench_N1.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cider.py needs a CUDA device (there is no CPU path to measure)")
    from bench import ClockSampler
    from icei_b200 import bleu, cider, ops
    from oracle import cider as oracle_cider
    try:
        from pycocoevalcap.cider.cider import Cider
    except ImportError:
        Cider = None
    info = device_info()
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
        (mean, got), e2e = timed(lambda: cider.corpus_cider(refs, hyps))
        scorer = cider.CiderD(refs)
        (mean_d, got_d), reuse = timed(lambda: scorer.compute_score(hyps))
        pack = []
        for _ in range(args.repeat):
            t0 = time.perf_counter()
            bleu._pack(refs, hyps)
            pack.append(1e3 * (time.perf_counter() - t0))
        # each kernel alone, on the packed device corpus
        views, max_len, max_group, ref_off_h, _ = cider._upload(refs, hyps)
        hyp_tok, hyp_off, ref_tok, ref_off, ref_group = views
        err = torch.zeros(1, dtype=torch.int32, device=hyp_off.device)
        cap = cider._capacity(ref_off_h, 4)
        keys, counts = ops.cider_df(ref_tok, ref_off, ref_group, 4, max_len, max_group, cap, err)
        out = torch.empty(n, dtype=torch.float64, device=hyp_off.device)
        df_ms = event_ms(lambda: ops.cider_df(ref_tok, ref_off, ref_group, 4, max_len, max_group, cap, err),
                         args.launches)
        scores_ms = event_ms(lambda: ops.cider_scores(hyp_tok, hyp_off, ref_tok, ref_off, ref_group, 4, 6.0, max_len,
                                                      max_group, keys, counts, out=out), args.launches)
        clocks = clocks.stop()
        t0 = time.perf_counter()
        want_mean, want = oracle_cider.corpus_cider(refs, hyps)
        oracle_ms = 1e3 * (time.perf_counter() - t0)
        ok = agree(got, want) and agree(mean, want_mean) and mean_d == mean and np.array_equal(got_d, got)
        coco_ms = None
        if Cider is not None:
            gts = {j: [" ".join(map(str, r)) for r in rs] for j, rs in enumerate(refs)}
            res = {j: [" ".join(map(str, h))] for j, h in enumerate(hyps)}
            t0 = time.perf_counter()
            _, coco = Cider(n=4, sigma=6.0).compute_score(gts, res)
            coco_ms = 1e3 * (time.perf_counter() - t0)
            ok = ok and agree(got, coco)
        rows.append({"n_img": n, "refs_per_img": args.refs, "tokens": tokens, "table_slots": cap,
                     "e2e_ms": round(statistics.median(e2e), 3), "e2e_ms_min": round(min(e2e), 3),
                     "ciderd_ms": round(statistics.median(reuse), 3), "pack_ms": round(statistics.median(pack), 3),
                     "df_ms": round(df_ms, 4), "scores_ms": round(scores_ms, 4), "oracle_ms": round(oracle_ms, 1),
                     "coco_ms": None if coco_ms is None else round(coco_ms, 1),
                     "max_abs_diff": float(np.abs(got - want).max()), "agree": ok, "cider": mean,
                     "sm_clock_mhz": clocks.get("sm_mhz"), "sm_clock_max_mhz": clocks.get("sm_max_mhz"),
                     "clock_reasons": clocks.get("reasons")})
    line = json.dumps(dict({"bench": "CIDEr-D (n=4, sigma=6)"}, **info, corpora=rows))
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
