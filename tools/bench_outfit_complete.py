"""Outfit completion (OutfitCompleter) against what a user writes without it.  Stage 1 -- predict_missing and one top-k per missing
slot (topk_batched) -- is shared by both paths and timed on its own.  Stage 2 is timed per path: OutfitCompleter.complete_local, and
the baseline, which builds every combination in torch, runs the model's autograd forward in blocks of `chunk` rows, computes the
errors in torch and takes torch.topk.  One JSON line per case.

Cases: embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)) with slots 1 and 2 missing at depth 16 (256 combinations per
outfit), Q = 128 and 1024, bf16 and fp32-parity engines, 1 M-row bf16 catalogs; the polyvore-shaped model (8 slots x 512,
10 x Linear(4096, 4096)) in bf16 with slots 1, 2 and 3 missing at depth 8 (512 combinations), Q = 256.  The paths alternate in one
process after a warm-up of both, timed with CUDA events around whole calls.  Their outputs are compared in the same run: the
largest relative difference of the k returned errors, and the ids that differ where the baseline's neighbouring errors are not a
near-tie (within the engine's tolerance).  The card's name and power limit are read in the same run.

    python tools/bench_outfit_complete.py [--reps 3] [--out profiles/r08_outfit_complete.jsonl]
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


def baseline(model, outfits, slots, cand, cats, E, depth, k, block):
    """Every combination of every outfit (all outfits miss the same slots) built in torch, the autograd forward in blocks of `block`
    rows, errors in torch, torch.topk per outfit; returns (err [Q, k], ids [Q, k, S])."""
    Q, S = outfits.shape[0], outfits.shape[1] // E
    C = depth ** len(slots)
    dev = outfits.device
    errs = []
    for p0 in range(0, Q * C, block):
        p = torch.arange(p0, min(p0 + block, Q * C), device=dev)
        q, c = p // C, p % C
        x = outfits[q].clone()
        for j, s in enumerate(slots):
            ids = cand[q, s, (c // depth ** j) % depth]
            x[:, s * E:(s + 1) * E] = cats[s][ids].float()
        with torch.no_grad():
            y = model(x)
        errs.append(((y - x) ** 2).sum(1))
    err = torch.cat(errs).view(Q, C)
    e, c = torch.topk(err, k, dim=1, largest=False)
    ids = torch.full((Q, k, S), -1, dtype=torch.int64, device=dev)
    for j, s in enumerate(slots):
        ids[:, :, s] = torch.gather(cand[:, s], 1, (c // depth ** j) % depth)
    return e, ids


def compare(e0, i0, e1, i1, rtol):
    """(largest relative difference of the returned errors, ids differing where the baseline's neighbours are further apart than
    the engine's tolerance)."""
    e0, e1 = e0.double().cpu(), e1.double().cpu()
    rel = ((e0 - e1).abs() / e0.abs().clamp_min(1e-30)).max().item()
    gap = torch.full_like(e0, float("inf"))
    d = e0[:, 1:] - e0[:, :-1]
    gap[:, 1:] = torch.minimum(gap[:, 1:], d)
    gap[:, :-1] = torch.minimum(gap[:, :-1], d)
    clear = gap > 4 * rtol * e0.abs()
    differ = (i0.cpu() != i1.cpu()).any(2)
    return rel, int((differ & clear).sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool import OutfitCompleter
    dev = torch.device("cuda", 0)
    name = card()
    E, N, k, chunk = 512, 1_000_000, 10, 8192
    g = torch.Generator(device=dev).manual_seed(0)
    out = open(args.out, "a") if args.out else None
    cases = [("embedding", 3, 1536, "bf16", 128, [1, 2], 16), ("embedding", 3, 1536, "bf16", 1024, [1, 2], 16),
             ("embedding", 3, 1536, "fp32", 128, [1, 2], 16), ("embedding", 3, 1536, "fp32", 1024, [1, 2], 16),
             ("polyvore", 8, 4096, "bf16", 256, [1, 2, 3], 8)]
    cats_for = {}
    for shape, S, z, engine, Q, slots, depth in cases:
        if (shape, S) not in cats_for:
            cats_for.clear()
            torch.cuda.empty_cache()
            cats_for[(shape, S)] = [torch.rand((N, E), generator=g, device=dev).to(torch.bfloat16) if s in slots else None
                                    for s in range(S)]
        cats = cats_for[(shape, S)]
        model = model_for(S, E, z, engine, dev)
        outfits = torch.rand((Q, S * E), generator=g, device=dev)
        missing = torch.zeros((Q, S), dtype=torch.bool, device=dev)
        missing[:, slots] = True
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=chunk)
        C = depth ** len(slots)
        box = {}

        def stage1():
            box["cand"] = comp.candidates(outfits, missing)

        def ours():
            box["ours"] = comp.complete_local(outfits, missing, box["cand"])

        def theirs():
            box["theirs"] = baseline(model, outfits, slots, box["cand"], cats, E, depth, k, chunk)
        stage1(); ours(); theirs()                         # warm-up of every path at this shape
        t1, t_c, t_b = [], [], []
        for _ in range(args.reps):
            t1.append(timed(stage1))
            t_c.append(timed(ours))
            t_b.append(timed(theirs))
        o_e, o_i = box["ours"]
        b_e, b_i = box["theirs"]
        rel, far = compare(b_e, b_i, o_e, o_i, RTOL[engine])
        line = {"model": "%s (io %d, 10 x %d^2)" % (shape, S * E, z), "engine": engine, "Q": Q, "missing": slots, "depth": depth,
                "combinations": Q * C, "catalog_rows": N, "catalog_dtype": "bf16", "chunk": chunk, "k": k,
                "ms_stage1_min": round(min(t1), 3), "ms_stage2_completer_min": round(min(t_c), 3),
                "ms_stage2_torch_min": round(min(t_b), 3), "ms_stage2_completer_median": round(statistics.median(t_c), 3),
                "ms_stage2_torch_median": round(statistics.median(t_b), 3), "stage2_torch_over_completer": round(min(t_b) / min(t_c), 3),
                "M_combinations_per_s_completer": round(Q * C / min(t_c) / 1e3, 3),
                "M_combinations_per_s_torch": round(Q * C / min(t_b) / 1e3, 3),
                "max_rel_err_diff": rel, "ids_differing_beyond_near_tie": far, "reps": args.reps, "card": name}
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()
        del comp, model, outfits, box
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
