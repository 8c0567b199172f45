#!/usr/bin/env python
"""Several styles per image in one beam search: ``sample_batch(..., mode=[style per image])`` against one single-style
``sample_batch`` per style, on one GPU.

    python bench_styles.py [--reps 40] [--json PATH]

Weights: configs[1] widths (V=10000, H=F=512, E=300), reference init + the decode recipe of bench_decode.py
(C.weight x30, C.bias[<end>] = +2) so captions end at varied lengths.  Workloads, k=5, feed_image=True:
  demo   one image x 4 styles (the demo back end's four captions per upload)
  batch  256 images x 4 styles
  cap    1..12 images x 4 styles (20..240 rows) on the few-row kernels vs the GEMM path: where the mixed few-row
         cap (decode.STYLES_SKINNY_MAX_ROWS) belongs
Both forms are timed in the same process, alternating, with the host clock around calls that end in a device
synchronise (the ids are read back).  The decode weights (~35 MB) stay in the 126 MB L2 across calls, as they do when a
server answers request after request: the numbers are for that regime.  The mixed and per-style ids are checked equal
in the same run.  Weight bytes per decode step are arithmetic from the shapes, not measurements."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
V, E, H, F = 10000, 300, 512, 512
K = 5


def sharpen(dec):
    import torch
    with torch.no_grad():
        dec.C.weight.mul_(30.0)
        dec.C.bias[2] = 2.0


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0].strip() if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def step_weight_bytes(n_styles, mixed):
    """fp32 weight bytes one decode step reads on the few-row path: collapsed chain Wc/bc per style, W_hh/b_hh, C/b_C;
    one mixed step reads the shared W_hh and C once, n single-style steps read them n times."""
    wc = (4 * H * E + 4 * H) * 4
    shared = (4 * H * H + 4 * H + V * H + V) * 4
    return n_styles * wc + shared if mixed else n_styles * (wc + shared)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--json", default=None, help="also write the rows to this file")
    args = ap.parse_args()
    import torch
    import icei_b200 as sn
    from icei_b200 import decode
    if not torch.cuda.is_available():
        raise SystemExit("bench_styles.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    gpu = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit()}
    print(json.dumps(gpu), flush=True)
    torch.manual_seed(0)
    dec = sn.DecoderFactoredLSTM(E, H, F, V, 1, dropout=0.5)
    sharpen(dec)
    dec = dec.to(dev).eval()
    styles = list(sn.STYLES)
    S = len(styles)
    g = torch.Generator().manual_seed(1)
    rows = []

    def run_mixed(x):
        n = x.shape[0]
        return dec.sample_batch(x.repeat_interleave(S, 0), 1, 2, k=K, mode=styles * n, feed_image=True)

    def run_four(x):
        per = [dec.sample_batch(x, 1, 2, k=K, mode=s, feed_image=True) for s in styles]
        return [per[j % S][j // S] for j in range(S * x.shape[0])]          # the mixed call's order: image, style

    def compare(name, x, reps):
        got_m, got_f = run_mixed(x), run_four(x)
        same = len(got_m) == len(got_f) and all(torch.equal(a, b) for a, b in zip(got_m, got_f))
        for _ in range(2):                  # warm-up: the 2nd call of a decode session captures its graphs
            run_mixed(x)
            run_four(x)
        t = {"mixed": 0.0, "four": 0.0}
        for _ in range(reps):               # alternate the two forms
            for key, fn in (("mixed", run_mixed), ("four", run_four)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(x)                       # ends in a device->host copy of the ids (a synchronise)
                t[key] += time.perf_counter() - t0
        n = x.shape[0]
        lens = sorted({int(a.shape[1]) for a in got_m})
        for key in ("mixed", "four"):
            ms = 1e3 * t[key] / reps
            row = {"workload": name, "form": key, "images": n, "styles": S, "k": K, "rows": n * S * K,
                   "ms_per_request": ms, "captions_per_s": n * S / (ms / 1e3),
                   "step_weight_MB_few_row": step_weight_bytes(S, key == "mixed") / 1e6,
                   "ids_identical": same, "caption_lengths": [lens[0], lens[-1]], "reps": reps,
                   "weights": "L2-resident across calls", **gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
        return same

    ok = compare("demo_1x4", torch.randn(1, E, generator=g).to(dev), args.reps)
    ok &= compare("batch_256x4", torch.randn(256, E, generator=g).to(dev), max(3, args.reps // 8))
    # where the mixed few-row path stops paying: the same requests forced onto each path
    cap = decode.STYLES_SKINNY_MAX_ROWS[0]
    for n in (1, 2, 4, 6, 8, 10, 12):
        x = torch.randn(n, E, generator=g).to(dev)
        res = {}
        for path, lim in (("few_row", 10 ** 6), ("gemm", 0)):
            decode.STYLES_SKINNY_MAX_ROWS[0] = lim
            dec.__dict__.pop("_decode_sessions", None)
            for _ in range(3):
                ids = run_mixed(x)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.reps):
                run_mixed(x)
            res[path] = (1e3 * (time.perf_counter() - t0) / args.reps, ids)
        decode.STYLES_SKINNY_MAX_ROWS[0] = cap
        dec.__dict__.pop("_decode_sessions", None)
        same = all(torch.equal(a, b) for a, b in zip(res["few_row"][1], res["gemm"][1]))
        row = {"workload": "cap_sweep", "images": n, "styles": S, "k": K, "rows": n * S * K,
               "few_row_ms": res["few_row"][0], "gemm_ms": res["gemm"][0], "ids_identical": same,
               "cap_rows": cap, **gpu}
        rows.append(row)
        print(json.dumps(row), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not ok:
        raise SystemExit("mixed-style and per-style ids differ")


if __name__ == "__main__":
    main()
