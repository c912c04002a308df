"""Filtered complementarity top-k against the unfiltered call: one JSON line per (catalog dtype, path, Q, filter).

Filters: an all-ones mask, 50 % and 1 % random masks, own-item exclusion (query q excludes global row q: n_exclude = 1) and
n_exclude = 256 random rows per query.  Each filtered call alternates with the unfiltered one (the old entry point) in the same
process on the same catalog, after a warm-up of both, timed with CUDA events around the whole call (the batched call includes
its device-to-host read and any fallback sweeps).  The sweep runs at Q = 1 and 4, the tensor-core batched path at Q = 64 and
1024.  The catalog (10 M x 512 by default: 10 GB bf16 / 20 GB fp32) is far larger than the 126 MB L2, so every call reads it
from HBM.

    python tools/bench_filtered_topk.py [--rows 10000000] [--E 512] [--k 10] [--reps 5] [--out FILE.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mui-deepautoencoder_b200"))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name(0)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--E", type=int, default=512)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dtypes", type=str, default="bf16,fp32")
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool.inference import ComplementarityScorer
    dev = torch.device("cuda", 0)
    name = card()
    n, E, k = args.rows, args.E, args.k
    g = torch.Generator(device=dev).manual_seed(0)
    base = torch.rand((n, E), generator=g, device=dev)
    masks = {"all-ones mask": torch.ones(n, dtype=torch.bool, device=dev),
             "50% mask": torch.rand(n, generator=g, device=dev) < 0.5,
             "1% mask": torch.rand(n, generator=g, device=dev) < 0.01}
    out = open(args.out, "a") if args.out else None
    for dtype in args.dtypes.split(","):
        cat = base.to(torch.bfloat16) if dtype == "bf16" else base
        unf = ComplementarityScorer(cat, E, "sqerr", k)
        scorers = {f: ComplementarityScorer(cat, E, "sqerr", k, allowed=m) for f, m in masks.items()}
        for path, Qs in (("sweep", (1, 4)), ("batched", (64, 1024))):
            for Q in Qs:
                q = torch.rand((Q, E), generator=g, device=dev)
                own = torch.arange(Q, dtype=torch.int64, device=dev).view(Q, 1)
                ex256 = torch.randint(0, n, (Q, 256), generator=g, device=dev)
                cases = [(f, sc, None) for f, sc in scorers.items()]
                cases += [("own-item exclusion (n_exclude = 1)", unf, own), ("n_exclude = 256", unf, ex256)]
                call = (lambda sc, ex: sc.topk_local(q, exclude=ex)) if path == "sweep" else \
                    (lambda sc, ex: sc.topk_local_batched(q, exclude=ex))
                for f, sc, ex in cases:
                    call(unf, None)
                    call(sc, ex)                              # warm-up of both at this shape
                    t0, t1, fb = [], [], 0
                    for _ in range(args.reps):
                        t0.append(timed(lambda: call(unf, None)))
                        t1.append(timed(lambda: call(sc, ex)))
                        if path == "batched":
                            fb = max(fb, sc.last_fallbacks)
                    line = {"catalog": "%d x %d %s" % (n, E, dtype), "metric": "sqerr", "path": path, "Q": Q, "k": k,
                            "filter": f, "ms_unfiltered_min": round(min(t0), 3), "ms_filtered_min": round(min(t1), 3),
                            "ms_unfiltered_median": round(statistics.median(t0), 3),
                            "ms_filtered_median": round(statistics.median(t1), 3),
                            "filtered_over_unfiltered_min": round(min(t1) / min(t0), 4),
                            "spread_unfiltered": round(max(t0) / min(t0), 4), "reps": args.reps, "card": name}
                    if path == "batched":
                        line["last_fallbacks_filtered"] = fb
                    s = json.dumps(line)
                    print(s, flush=True)
                    if out:
                        out.write(s + "\n")
                        out.flush()
        del unf, scorers, cat
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
