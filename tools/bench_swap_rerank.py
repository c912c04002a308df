"""Swap re-ranking over per-outfit candidate lists (SwapScorer.rerank_local) against what the per-outfit API allows: a loop of
SwapScorer.topk_local calls, one per outfit, each on that outfit's listed rows gathered into a catalog of m rows.  One JSON line
per case.

Cases: embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)) with the bf16 and the fp32-parity engines at
Q = 1024 outfits x m = 100 ids (retrieve-then-re-rank), Q = 10 000 x m = 4 (fill-in-the-blank questions), Q = 64 x m = 16 384
(large lists: compare pairs/s with the full-catalog sweep, timed in the same run on the same model), and the polyvore-shaped
model (8 slots x 512, 10 x Linear(4096, 4096), bf16) at Q = 1024 x m = 100.  Ids are drawn from a 1 M x 512 fp32 catalog.
The two paths alternate in one process after a warm-up of both at every shape, timed with CUDA events around whole calls (the
rerank call includes its one host synchronisation).  Their outputs are compared in the same run: ids equal apart from near-ties,
errors within the engine's tolerance.

    python tools/bench_swap_rerank.py [--reps 3] [--out profiles/r05_swap_rerank.jsonl]
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
RTOL = {"bf16": 1e-2, "fp32": 1e-5}


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


def model_for(S, E, z, engine, dev):
    from codae.model import EmbeddingDenoisingAutoencoder
    torch.manual_seed(S)
    m = EmbeddingDenoisingAutoencoder(S * E, z, E, 4, 4, False)
    return m.to(dev).set_compute_dtype(engine)


def compare(s0, i0, s1, i1, rtol):
    """(fraction of equal ids, ids that differ beyond a near-tie, largest relative error difference) of two [Q, k] results."""
    s0, i0, s1, i1 = (t.double().cpu() if t.is_floating_point() else t.cpu() for t in (s0, i0, s1, i1))
    used = (i0 >= 0) & (i1 >= 0)                        # unused slots are (+inf, -1) in both
    rel = ((s0 - s1).abs() / s0.abs().clamp_min(1e-30))[used].max().item()
    kth = torch.where(used, s0, torch.zeros_like(s0)).max(dim=1, keepdim=True).values
    differ = i0 != i1
    # an id that differs is a near-tie when its error lies within the tolerance of the other list's error at that place
    far = differ & ~(used & ((s0 - s1).abs() <= rtol * kth))
    return (1 - differ.double().mean().item()), int(far.sum().item()), rel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool.inference import SwapScorer
    dev = torch.device("cuda", 0)
    name = card()
    E, n, k, slot = 512, args.rows, args.k, 1
    g = torch.Generator(device=dev).manual_seed(0)
    cat = torch.rand((n, E), generator=g, device=dev)
    out = open(args.out, "a") if args.out else None
    cases = [("embedding", 3, 1536, "bf16", 1024, 100), ("embedding", 3, 1536, "fp32", 1024, 100),
             ("embedding", 3, 1536, "bf16", 10_000, 4), ("embedding", 3, 1536, "bf16", 64, 16_384),
             ("polyvore", 8, 4096, "bf16", 1024, 100)]
    for shape, S, z, engine, Q, m in cases:
        model = model_for(S, E, z, engine, dev)
        outfits = torch.rand((Q, S * E), generator=g, device=dev)
        cand = torch.randint(0, n, (Q, m), generator=g, device=dev)
        sc = SwapScorer(model, cat, E, k=k)
        rows = torch.empty((m, E), device=dev)
        loop_sc = SwapScorer(model, rows, E, k=k)

        def rerank():
            return sc.rerank_local(outfits, slot, cand)

        def loop():
            s = torch.empty((Q, k), device=dev)
            i = torch.empty((Q, k), dtype=torch.int64, device=dev)
            for q in range(Q):
                torch.index_select(cat, 0, cand[q], out=rows)
                sq, iq = loop_sc.topk_local(outfits[q], slot)
                s[q] = sq
                i[q] = cand[q][iq.clamp_min(0)].masked_fill(iq < 0, -1)
            return s, i
        r_s, r_i = (t.clone() for t in rerank())
        l_s, l_i = loop()                                  # warm-up of both at this shape
        t_r, t_l = [], []
        for _ in range(args.reps):
            t_r.append(timed(rerank))
            t_l.append(timed(loop))
        same, far, rel = compare(l_s, l_i, r_s, r_i, RTOL[engine])
        line = {"model": "%s (io %d, 10 x %d^2)" % (shape, S * E, z), "engine": engine, "Q": Q, "m": m, "k": k,
                "catalog": "%d x %d fp32" % (n, E), "chunk": sc.chunk,
                "ms_rerank_min": round(min(t_r), 3), "ms_loop_min": round(min(t_l), 3),
                "ms_rerank_median": round(statistics.median(t_r), 3), "ms_loop_median": round(statistics.median(t_l), 3),
                "loop_over_rerank": round(min(t_l) / min(t_r), 3),
                "M_pairs_per_s_rerank": round(Q * m / min(t_r) / 1e3, 3), "M_pairs_per_s_loop": round(Q * m / min(t_l) / 1e3, 3),
                "ids_equal_fraction": round(same, 6), "ids_differing_beyond_near_tie": far, "max_rel_error_diff": rel,
                "reps": args.reps, "card": name}
        if m >= 8192:                                      # the full-catalog sweep on the same model: swaps/s for reference
            full = lambda: sc.topk_local(outfits[0], slot)
            full()
            t_f = min(timed(full) for _ in range(args.reps))
            line["ms_full_catalog_sweep_min"] = round(t_f, 3)
            line["M_swaps_per_s_full_catalog_sweep"] = round(n / t_f / 1e3, 3)
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()
        del sc, loop_sc, model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
