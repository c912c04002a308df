"""Outfit revision (OutfitCompleter.revise_candidates / revise_local) against what a user writes without it: for every slot s,
predict_slot, a top-k of slot s's catalog (topk_batched) and SwapScorer.rerank_local over those candidates; then the autograd
forward of the outfits as given for the base error and a torch merge of the S lists that keeps the swaps below it.  Stage 1 (the
candidates) and stage 2 (the swap errors and the ranking) are timed on their own for both paths.  One JSON line per case.

Cases: embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)) at Q = 128, 1024 and 10 000 outfits, bf16 and fp32-parity
engines; the polyvore-shaped model (8 slots x 512, 10 x Linear(4096, 4096)) in bf16 at Q = 256 and 1024; depth 16, k = 10,
1 M-row bf16 catalogs, chunk 8192.  The paths alternate in one process after a warm-up of both, timed with CUDA events around whole
calls.  Both stage 2s score the candidates of revise_candidates, so their outputs are compared in the same run: the largest relative
difference of the base errors and of the listed swap errors, and the listed (slot, id) that differ where the baseline's neighbouring
errors are not a near-tie (within the engine's tolerance).  Stage 1's ids are compared too.  The card's name, power limit and
maximum SM clock are read in the same run.

    python tools/bench_outfit_revise.py [--reps 3] [--out profiles/r10_outfit_revise.jsonl]
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


def baseline_stage1(model, outfits, scorers, E):
    """S x (predict_slot -> topk_batched): [Q, S, depth] ids."""
    from codae.tool.inference import predict_slot
    return torch.stack([sc.topk_batched(predict_slot(model, outfits, s, E))[1] for s, sc in enumerate(scorers)], 1)


def baseline_stage2(model, outfits, cand, swappers, k, block):
    """S SwapScorer.rerank_local calls, the outfits' own error by the autograd forward in blocks, then a torch merge of the S lists
    by (error, s depth + rank) cut at the base: (base [Q], err [Q, k], slot [Q, k], ids [Q, k])."""
    Q, S, depth = cand.shape
    errs, ids = zip(*[sw.rerank_local(outfits, s, cand[:, s].contiguous()) for s, sw in enumerate(swappers)])
    with torch.no_grad():
        base = torch.cat([((model(outfits[b:b + block]) - outfits[b:b + block]) ** 2).sum(1) for b in range(0, Q, block)])
    err = torch.cat(errs, 1)
    idx = torch.cat(ids, 1)
    slot = torch.arange(S, device=outfits.device).repeat_interleave(depth).expand(Q, -1)
    e, order = torch.sort(torch.where(torch.isnan(err), float("inf"), err), dim=1, stable=True)
    e, order = e[:, :k], order[:, :k]
    better = e < base.unsqueeze(1)
    return (base, torch.where(better, e, float("inf")), torch.where(better, torch.gather(slot, 1, order), -1),
            torch.where(better, torch.gather(idx, 1, order), -1))


def compare(ref, got, rtol):
    """(largest relative base difference, largest relative listed-error difference, listed entries that differ where the
    baseline's neighbouring errors are further apart than the engine's tolerance)."""
    rb, re_, rs, ri = (t.cpu() for t in ref)
    gb, ge, gs, gi = (t.cpu() for t in got)
    rel_b = ((rb.double() - gb.double()).abs() / rb.double().abs().clamp_min(1e-30)).max().item()
    both = torch.isfinite(re_) & torch.isfinite(ge)
    d = (re_.double() - ge.double()).abs() / re_.double().abs().clamp_min(1e-30)
    rel_e = d[both].max().item() if bool(both.any()) else 0.0
    e0 = torch.where(torch.isfinite(re_), re_, 1e30).double()
    gap = torch.full_like(e0, float("inf"))
    dd = e0[:, 1:] - e0[:, :-1]
    gap[:, 1:] = torch.minimum(gap[:, 1:], dd)
    gap[:, :-1] = torch.minimum(gap[:, :-1], dd)
    near_base = (rb.double().unsqueeze(1) - e0).abs() <= 4 * rtol * e0.abs()
    clear = (gap > 4 * rtol * e0.abs()) & ~near_base
    differ = (rs != gs) | (ri != gi)
    return rel_b, rel_e, int((differ & clear).sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool import ComplementarityScorer, OutfitCompleter, SwapScorer
    dev = torch.device("cuda", 0)
    name = card()
    E, N, k, chunk, depth = 512, 1_000_000, 10, 8192, 16
    g = torch.Generator(device=dev).manual_seed(0)
    out = open(args.out, "a") if args.out else None
    cases = [("embedding", 3, 1536, "bf16", 128), ("embedding", 3, 1536, "bf16", 1024), ("embedding", 3, 1536, "bf16", 10_000),
             ("embedding", 3, 1536, "fp32", 128), ("embedding", 3, 1536, "fp32", 1024), ("embedding", 3, 1536, "fp32", 10_000),
             ("polyvore", 8, 4096, "bf16", 256), ("polyvore", 8, 4096, "bf16", 1024)]
    cats_for = {}
    for shape, S, z, engine, Q in cases:
        if (shape, S) not in cats_for:
            cats_for.clear()
            torch.cuda.empty_cache()
            cats_for[(shape, S)] = [torch.rand((N, E), generator=g, device=dev).to(torch.bfloat16) for _ in range(S)]
        cats = cats_for[(shape, S)]
        model = model_for(S, E, z, engine, dev)
        outfits = torch.rand((Q, S * E), generator=g, device=dev)
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=chunk)
        scorers = [ComplementarityScorer(c, E, k=depth) for c in cats]
        swappers = [SwapScorer(model, c, E, k=depth, chunk=chunk) for c in cats]
        box = {}

        def ours1():
            box["cand"] = comp.revise_candidates(outfits)

        def theirs1():
            box["cand_b"] = baseline_stage1(model, outfits, scorers, E)

        def ours2():
            box["ours"] = comp.revise_local(outfits, box["cand"])

        def theirs2():
            box["theirs"] = baseline_stage2(model, outfits, box["cand"], swappers, k, chunk)
        ours1(); theirs1(); ours2(); theirs2()             # warm-up of every path at this shape
        t1, b1, t2, b2 = [], [], [], []
        for _ in range(args.reps):
            t1.append(timed(ours1))
            b1.append(timed(theirs1))
            t2.append(timed(ours2))
            b2.append(timed(theirs2))
        rel_b, rel_e, far = compare(box["theirs"], box["ours"], RTOL[engine])
        rows = Q * (1 + S * depth)
        line = {"model": "%s (io %d, 10 x %d^2)" % (shape, S * E, z), "engine": engine, "Q": Q, "slots": S, "depth": depth, "k": k,
                "grid_rows": rows, "catalog_rows": N, "catalog_dtype": "bf16", "chunk": chunk,
                "ms_stage1_revise_min": round(min(t1), 3), "ms_stage1_by_hand_min": round(min(b1), 3),
                "ms_stage2_revise_min": round(min(t2), 3), "ms_stage2_by_hand_min": round(min(b2), 3),
                "ms_stage2_revise_median": round(statistics.median(t2), 3), "ms_stage2_by_hand_median": round(statistics.median(b2), 3),
                "stage2_by_hand_over_revise": round(min(b2) / min(t2), 3),
                "total_by_hand_over_revise": round((min(b1) + min(b2)) / (min(t1) + min(t2)), 3),
                "M_rows_per_s_stage2_revise": round(rows / min(t2) / 1e3, 3),
                "listed_swaps_per_outfit": round(float(torch.isfinite(box["ours"][1]).sum()) / Q, 3),
                "stage1_ids_equal_fraction": round(float((box["cand"] == box["cand_b"]).float().mean()), 5),
                "max_rel_base_diff": rel_b, "max_rel_err_diff": rel_e, "entries_differing_beyond_near_tie": far, "reps": args.reps,
                "card": name}
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()
        del comp, model, outfits, box, scorers, swappers
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
