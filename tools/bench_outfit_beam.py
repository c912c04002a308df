"""Outfit completion by beam search (OutfitCompleter.complete_beam_local) where exhaustive completion still runs, and where it does not.
Stage 1 -- predict_missing and one top-k per missing slot -- is shared by every path and timed on its own.  One JSON line per case.

"exhaustive" cases: embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)), slots 1 and 2 missing at depth 16, Q = 1024,
bf16 and fp32-parity engines.  The beam at W = 1, 4 and 16 alternates with complete_local in one process; for each W the line holds
both times and the agreement with exhaustive search: the share of outfits whose best combination is the same, and the mean overlap
of the top-k id sets (k = min(10, W)).  W = 16 = depth^(m - 1) prunes nothing.

"beam" cases: the polyvore-shaped model (8 slots x 512, 10 x Linear(4096, 4096)) in bf16, slots 1..7 missing at depth 16 (16^7
combinations, past complete's cap), W = 4, 16, 64, Q = 256.  Reported: DAE rows per second of the beam against SwapScorer.rerank_local
on the same model (128 candidates per outfit); baseline 1, the same beam written in torch over the model's forward (alternating, with
the outputs compared: largest relative difference of the returned errors and ids differing beyond a near-tie); baseline 2, what a
user can run today, complete_local at depth 3 (3^7 = 2187 combinations per outfit).

Timed with CUDA events around whole calls after a warm-up of every path; the card's name, power limit and max SM clock are read in
the same run.

    python tools/bench_outfit_beam.py [--reps 3] [--out profiles/r09_outfit_beam.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mui-deepautoencoder_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_outfit_complete import RTOL, card, compare, model_for, timed  # noqa: E402


def torch_beam(model, outfits, slots, cand, cats, E, depth, W, k, block):
    """The beam in torch: per level every child of every kept partial outfit built in torch (later missing slots zero), the model's
    forward in blocks of `block` rows, partial errors over the visible columns, torch.topk per outfit.  (err [Q, k], ids [Q, k, S])."""
    Q, S = outfits.shape[0], outfits.shape[1] // E
    dev = outfits.device
    beam = torch.zeros((Q, 1), dtype=torch.int64, device=dev)
    for j, s in enumerate(slots):
        kids = (beam.unsqueeze(2) + torch.arange(depth, device=dev) * depth ** j).view(Q, -1)
        n_kids = kids.shape[1]
        vis = torch.ones(S * E, device=dev)
        for s2 in slots[j + 1:]:
            vis[s2 * E:(s2 + 1) * E] = 0
        errs = []
        for p0 in range(0, Q * n_kids, block):
            p = torch.arange(p0, min(p0 + block, Q * n_kids), device=dev)
            q, c = p // n_kids, kids.view(-1)[p]
            x = outfits[q].clone()
            for jj, ss in enumerate(slots):
                if jj <= j:
                    x[:, ss * E:(ss + 1) * E] = cats[ss][cand[q, ss, (c // depth ** jj) % depth]].float()
                else:
                    x[:, ss * E:(ss + 1) * E] = 0
            with torch.no_grad():
                y = model(x)
            errs.append((((y - x) ** 2) * vis).sum(1))
        err = torch.cat(errs).view(Q, n_kids)
        e, idx = torch.topk(err, min(W, n_kids), dim=1, largest=False)
        beam = torch.gather(kids, 1, idx)
    ids = torch.full((Q, k, S), -1, dtype=torch.int64, device=dev)
    for j, s in enumerate(slots):
        ids[:, :, s] = torch.gather(cand[:, s], 1, (beam[:, :k] // depth ** j) % depth)
    return e[:, :k], ids


def agreement(b_ids, x_ids):
    """(share of outfits whose best combination equals exhaustive's, mean top-k id-set overlap) for [Q, k, S] ids."""
    best = (b_ids[:, 0] == x_ids[:, 0]).all(1).double().mean().item()
    eq = (b_ids.unsqueeze(2) == x_ids.unsqueeze(1)).all(3)             # [Q, k, k]
    overlap = eq.any(2).double().sum(1).div(b_ids.shape[1]).mean().item()
    return round(best, 4), round(overlap, 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool import OutfitCompleter, SwapScorer
    dev = torch.device("cuda", 0)
    name = card()
    E, N, chunk = 512, 1_000_000, 8192
    g = torch.Generator(device=dev).manual_seed(0)
    out = open(args.out, "a") if args.out else None

    def emit(line):
        line.update(reps=args.reps, card=name)
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    # where exhaustive completion still runs
    S, z, Q, slots, depth = 3, 1536, 1024, [1, 2], 16
    cats = [torch.rand((N, E), generator=g, device=dev).to(torch.bfloat16) if s in slots else None for s in range(S)]
    for engine in ("bf16", "fp32"):
        model = model_for(S, E, z, engine, dev)
        outfits = torch.rand((Q, S * E), generator=g, device=dev)
        missing = torch.zeros((Q, S), dtype=torch.bool, device=dev)
        missing[:, slots] = True
        for W in (1, 4, 16):
            k = min(10, W)
            comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=chunk)
            box = {}

            def stage1():
                box["cand"] = comp.candidates(outfits, missing)

            def exhaustive():
                box["x"] = [t.clone() for t in comp.complete_local(outfits, missing, box["cand"])]

            def beam():
                box["b"] = [t.clone() for t in comp.complete_beam_local(outfits, missing, box["cand"], W)]
            stage1(); exhaustive(); beam()
            t1, tx, tb = [], [], []
            for _ in range(args.reps):
                t1.append(timed(stage1))
                tx.append(timed(exhaustive))
                tb.append(timed(beam))
            best, overlap = agreement(box["b"][1], box["x"][1])
            rows = Q * depth * sum(min(W, depth ** j) for j in range(len(slots)))
            emit({"case": "exhaustive", "model": "embedding (io 1536, 10 x 1536^2)", "engine": engine, "Q": Q, "missing": slots,
                  "depth": depth, "W": W, "k": k, "chunk": chunk, "catalog_rows": N, "catalog_dtype": "bf16",
                  "ms_stage1_min": round(min(t1), 3), "ms_beam_min": round(min(tb), 3), "ms_beam_median": round(statistics.median(tb), 3),
                  "ms_exhaustive_min": round(min(tx), 3), "ms_exhaustive_median": round(statistics.median(tx), 3),
                  "beam_rows": rows, "exhaustive_rows": Q * depth ** len(slots),
                  "best_equal_share": best, "topk_overlap": overlap})
            del comp, box
        del model
        torch.cuda.empty_cache()
    del cats
    torch.cuda.empty_cache()

    # where it does not: the polyvore shape, 7 of 8 slots missing
    S, z, Q, slots, depth = 8, 4096, 256, list(range(1, 8)), 16
    cats = [torch.rand((N, E), generator=g, device=dev).to(torch.bfloat16) if s in slots else None for s in range(S)]
    model = model_for(S, E, z, "bf16", dev)
    outfits = torch.rand((Q, S * E), generator=g, device=dev)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=dev)
    missing[:, slots] = True
    base = OutfitCompleter(model, cats, E, depth=depth, k=10, chunk=chunk)
    cand = base._beam_candidates(outfits, missing)          # complete_beam's stage 1, timed alone
    t1 = [timed(lambda: base._beam_candidates(outfits, missing)) for _ in range(args.reps)]
    d3 = OutfitCompleter(model, cats, E, depth=3, k=10, chunk=chunk)
    cand3 = cand[:, :, :3].contiguous()
    swap = SwapScorer(model, cats[1], E, k=10, chunk=chunk)
    swap_cand = torch.randint(0, N, (Q, 128), generator=g, device=dev)
    box = {}

    def rerank():
        box["r"] = swap.rerank_local(outfits, 1, swap_cand)

    def complete3():
        box["c3"] = d3.complete_local(outfits, missing, cand3)
    rerank(); complete3()
    t_sw = [timed(rerank) for _ in range(args.reps)]
    t_c3 = [timed(complete3) for _ in range(args.reps)]
    for W in (4, 16, 64):
        k = min(10, W)
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=chunk)

        def beam():
            box["b"] = [t.clone() for t in comp.complete_beam_local(outfits, missing, cand, W)]

        def theirs():
            box["t"] = torch_beam(model, outfits, slots, cand, cats, E, depth, W, k, chunk)
        beam(); theirs()
        tb, tt = [], []
        for _ in range(args.reps):
            tb.append(timed(beam))
            tt.append(timed(theirs))
        rel, far = compare(box["t"][0], box["t"][1], box["b"][0], box["b"][1], RTOL["bf16"])
        rows = Q * depth * sum(min(W, depth ** j) for j in range(len(slots)))
        emit({"case": "beam", "model": "polyvore (io 4096, 10 x 4096^2)", "engine": "bf16", "Q": Q, "missing": slots, "depth": depth,
              "W": W, "k": k, "chunk": chunk, "catalog_rows": N, "catalog_dtype": "bf16", "ms_stage1_min": round(min(t1), 3),
              "ms_beam_min": round(min(tb), 3), "ms_beam_median": round(statistics.median(tb), 3),
              "ms_torch_beam_min": round(min(tt), 3), "torch_beam_over_beam": round(min(tt) / min(tb), 3),
              "beam_rows": rows, "M_rows_per_s_beam": round(rows / min(tb) / 1e3, 3),
              "M_rows_per_s_swap_rerank": round(Q * 128 / min(t_sw) / 1e3, 3),
              "ms_complete_depth3_min": round(min(t_c3), 3), "complete_depth3_rows": Q * 3 ** len(slots),
              "max_rel_err_diff_vs_torch": rel, "ids_differing_beyond_near_tie": far})
        del comp


if __name__ == "__main__":
    main()
