"""Batched complementarity top-k against the row sweep: one JSON line per (catalog dtype, metric, Q).

Both paths run in the same process on the same catalog, alternating call by call after a warm-up, timed with CUDA events
around each whole call (the batched call includes its one device-to-host read and any fallback sweeps).  The catalog
(10 M x 512 by default: 10 GB bf16 / 20 GB fp32) is far larger than the 126 MB L2, so every call reads it from HBM.

    python tools/bench_batched_topk.py [--rows 10000000] [--E 512] [--k 10] [--queries 1,16,64,256,1024,4096] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mui-deepautoencoder_b200"))

BF16_DENSE_PEAK = 2250e12      # NVIDIA HGX B200 data sheet, dense BF16, per GPU (a 1000 W card)


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
    ap.add_argument("--queries", type=str, default="1,16,64,256,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", type=str, default="bf16:sqerr,bf16:cosine,fp32:sqerr")
    args = ap.parse_args()
    from codae.tool.inference import ComplementarityScorer
    dev = torch.device("cuda", 0)
    name = card()
    n, E, k = args.rows, args.E, args.k
    g = torch.Generator(device=dev).manual_seed(0)
    base = torch.rand((n, E), generator=g, device=dev)
    for cfg in args.configs.split(","):
        dtype, metric = cfg.split(":")
        cat = base.to(torch.bfloat16) if dtype == "bf16" else base
        sc = ComplementarityScorer(cat, E, metric, k)
        for Q in [int(x) for x in args.queries.split(",")]:
            q = torch.rand((Q, E), generator=g, device=dev)
            sc.topk_local(q)
            sc.topk_local_batched(q)                      # warm-up of both paths at this shape
            t_sweep, t_tc, fallbacks = [], [], 0
            for _ in range(args.reps):
                t_sweep.append(timed(lambda: sc.topk_local(q)))
                t_tc.append(timed(lambda: sc.topk_local_batched(q)))
                fallbacks = max(fallbacks, sc.last_fallbacks)
            ms_sweep, ms_tc = min(t_sweep), min(t_tc)
            flop = 2.0 * Q * n * E
            print(json.dumps({"catalog": "%d x %d %s" % (n, E, dtype), "metric": metric, "Q": Q, "k": k,
                              "ms_sweep": round(ms_sweep, 3), "ms_batched": round(ms_tc, 3),
                              "speedup": round(ms_sweep / ms_tc, 2),
                              "batched_useful_tflops": round(flop / (ms_tc * 1e-3) / 1e12, 1),
                              "share_of_bf16_dense_peak": round(flop / (ms_tc * 1e-3) / BF16_DENSE_PEAK, 3),
                              "peak": "2250 TFLOP/s dense BF16 (B200 data sheet, 1000 W)",
                              "catalog_bytes_per_call": n * E * cat.element_size(),
                              "last_fallbacks": fallbacks, "reps": args.reps, "card": name}), flush=True)
        del sc, cat
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
