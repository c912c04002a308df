"""Stage IV: complementarity inference (README.md:14-16,30-32 of the reference names this entry point; the
script itself is absent there, the shipped logic is RankingLoss, codae/tool/metering.py:46-79).

For each query outfit: zero the requested slot, run the trained DAE, and rank the catalog items of that
category against the reconstructed slot (squared error by default, or cosine similarity), returning the
top-k.  The catalog is sharded by rows across ranks (torchrun), merged with an all-gather of k entries.

--mode swap scores every candidate SWAP by the reconstruction error of the whole swapped outfit instead
(candidate substituted into the slot, DAE forward per candidate; codae.tool.SwapScorer).

--mode rerank retrieves, then re-ranks: the top --rerank_depth M rows of the slot reading (--metric) for every outfit, then
those M candidates scored by swap error in one batched pass (SwapScorer.rerank); it prints the final k with their swap errors.

--exclude_own_item leaves out, for query q, catalog row q (the item outfit q already holds in the slot: a trained DAE
reconstructs it closely, and swapping it in is the identity swap); --allowed_rows PATH.npy restricts the results to the
global row ids stored there (int64).  Both filter inside the kernels, so k results come back whenever k rows are eligible.

--mode compat scores how well the items of the first --queries outfits go together (codae.tool.CompatibilityScorer): every slot
is hidden in turn and reconstructed; it prints each outfit's per-slot errors, their sum (lower: more compatible) and the slot of
largest error (the odd item out).  No catalog is built.  --compat_negatives also scores one shuffled outfit per query -- slot s
taken from a seeded permutation of all observations -- and adds the compatibility AUC of the real outfits against them.

--mode complete fills the slots listed by --missing (e.g. 1,2) of the first --queries outfits together
(codae.tool.OutfitCompleter): the best --complete_depth B rows per missing slot by --metric, then every combination of them
scored by the reconstruction error of the completed outfit; it prints the best k completions as ids [Q][k][S] (-1 in given slots)
with their errors [Q][k].  --exclude_own_item and --allowed_rows do not apply to this mode.  With --beam W the combinations
are searched by a beam of width W instead (OutfitCompleter.complete_beam: the missing slots filled one at a time, the best W
partial outfits kept after each), which has no cap on depth^#missing; the JSON then also holds "beam": W.

--mode revise asks of each of the first --queries outfits, complete as they are, which one item to replace and with what
(codae.tool.OutfitCompleter.revise): every slot is read with only that slot hidden, its best --complete_depth B catalog rows by
--metric are swapped in one at a time, and the swaps whose reconstruction error is below the outfit's own are ranked.  It prints
the outfit's error as "base" [Q] and the best k swaps as "errors", "slots" and "ids" [Q][k] (+inf / -1 where fewer swaps improve).
--exclude_own_item keeps each outfit's own items out of its candidates (outfit q holds row q of every slot's catalog);
--allowed_rows does not apply to this mode.
"""
import argparse
import json

import numpy as np
import torch
import yaml

import _common  # noqa: F401
from _common import init_distributed, synthetic_categories
from codae.dataset import ConcatenatedEmbeddingDataset
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool import load_dataset_of_embeddings
from codae.tool.inference import (CompatibilityScorer, ComplementarityScorer, OutfitCompleter, SwapScorer, compatibility_auc,
                                  predict_slot, shard_rows)


def parse():
    parser = argparse.ArgumentParser(description='Rank catalog items for a missing outfit slot.')
    parser.add_argument('--embedding_path', type=str, default=None)
    parser.add_argument('--config', type=str, required=True)
    parser.add_argument('--model_path', type=str, default=None)
    parser.add_argument('--slot', type=int, default=0)
    parser.add_argument('--k', type=int, default=10)
    parser.add_argument('--metric', type=str, default="sqerr", choices=["sqerr", "cosine"])
    parser.add_argument('--mode', type=str, default="slot", choices=["slot", "swap", "rerank", "compat", "complete",
                                                                                "revise"])
    parser.add_argument('--rerank_depth', type=int, default=50, help="rerank mode: stage-1 candidates per outfit (1..128)")
    parser.add_argument('--missing', type=str, default="1", help="complete mode: comma-separated slots to fill")
    parser.add_argument('--complete_depth', type=int, default=8,
                        help="complete mode: candidates per missing slot (1..128, depth^#missing <= 4096 without --beam); "
                             "revise mode: candidates per slot (1..128)")
    parser.add_argument('--beam', type=int, default=None,
                        help="complete mode: search by a beam of this width (k <= W <= 128) instead of every combination")
    parser.add_argument('--compute_dtype', '--dtype', dest="compute_dtype", type=str, default="fp32", choices=["fp32", "bf16", "fp32_simt"])
    parser.add_argument('--queries', type=int, default=4)
    parser.add_argument('--synthetic', type=int, default=0)
    parser.add_argument('--catalog_dtype', type=str, default="fp32", choices=["fp32", "bf16", "fp32_simt"])
    parser.add_argument('--exclude_own_item', action='store_true', help="query q never gets catalog row q back")
    parser.add_argument('--compat_negatives', action='store_true',
                        help="compat mode: also score one shuffled outfit per query and report the AUC")
    parser.add_argument('--allowed_rows', type=str, default=None, help=".npy of int64 global row ids that may be returned")
    return parser.parse_args()


def local_allowed(path, lo, n_local, device):
    """Mask of this rank's rows [lo, lo + n_local) from a file of global row ids (None without a file)."""
    if path is None:
        return None
    rows = torch.from_numpy(np.load(path).astype(np.int64).reshape(-1))
    rows = rows[(rows >= lo) & (rows < lo + n_local)] - lo
    mask = torch.zeros(n_local, dtype=torch.bool)
    mask[rows] = True
    return mask.to(device)


if __name__ == "__main__":
    args = parse()
    if args.mode == "rerank" and not 1 <= args.rerank_depth <= 128:
        raise SystemExit("--rerank_depth must lie in [1, 128]")
    if args.mode == "complete" and (args.exclude_own_item or args.allowed_rows):
        raise SystemExit("--exclude_own_item and --allowed_rows are not supported by --mode complete (completion takes no filters)")
    if args.mode == "revise" and args.allowed_rows:
        raise SystemExit("--allowed_rows is not supported by --mode revise (revision takes no allowed-row mask)")
    rank, world, device = init_distributed()
    with open(args.config, 'r') as stream:
        config = yaml.safe_load(stream)
    cats = config["DATASET"]["USED_CATEGORY"]
    E = config["DATASET"]["EMBEDDING_SIZE"]
    if args.synthetic > 0:
        dataset = ConcatenatedEmbeddingDataset.from_tensors(synthetic_categories(args.synthetic, len(cats), E, config["SEED"]), cats)
    else:
        dataset = load_dataset_of_embeddings(embedding_path=args.embedding_path, config=config, cache_dir="tmp/")
    torch.manual_seed(config["SEED"])
    model = EmbeddingDenoisingAutoencoder(io_size=E * len(cats), z_size=config["MODEL"]["Z_SIZE"], embedding_size=E,
                                          nb_input_layer=config["MODEL"]["NB_INPUT_LAYER"],
                                          nb_output_layer=config["MODEL"]["NB_OUTPUT_LAYER"],
                                          steep_layer_size=config["MODEL"]["STEEP_LAYER_SIZE"])
    if args.model_path:
        model.load_state_dict(torch.load(args.model_path, map_location="cpu"))
    model.to(device).set_compute_dtype(args.compute_dtype)
    if args.mode == "compat":
        compat = CompatibilityScorer(model, E)
        outfits = dataset.data[:args.queries].float().to(device).contiguous()
        err, score, odd = (t.clone() for t in compat.score(outfits))
        res = {"mode": "compat", "slots": compat.S, "score": score.cpu().tolist(), "slot_errors": err.cpu().tolist(),
               "odd_slot": odd.cpu().tolist()}
        if args.compat_negatives:
            # one negative per query: slot s of negative q is slot s of observation perm_s[q] (a seeded permutation per slot)
            g = torch.Generator().manual_seed(config["SEED"])
            neg = torch.empty_like(outfits)
            for s in range(compat.S):
                perm = torch.randperm(dataset.nb_observation, generator=g)[:outfits.shape[0]]
                neg[:, s * E:(s + 1) * E] = dataset.data[perm, s * E:(s + 1) * E].to(device)
            _, neg_score, _ = compat.score(neg)
            res["auc"] = compatibility_auc(score, neg_score)
        if rank == 0:
            print(json.dumps(res))
        raise SystemExit(0)
    lo, n_local = shard_rows(dataset.nb_observation, world, rank)
    if args.mode == "complete":
        slots = sorted({int(v) for v in args.missing.split(",")})
        S = len(cats)
        if not slots or not all(0 <= s < S for s in slots):
            raise SystemExit("--missing must list slots in [0, %d)" % S)
        cat_dtype = torch.bfloat16 if args.catalog_dtype == "bf16" else torch.float32
        catalogs = [dataset.data_per_category[s][lo:lo + n_local].to(device).to(cat_dtype).contiguous() if s in slots else None
                    for s in range(S)]
        comp = OutfitCompleter(model, catalogs, E, depth=args.complete_depth, k=args.k, metric=args.metric,
                               inv_scale=1.0 / dataset.scale, row_offsets=[lo] * S)
        outfits = dataset.data[:args.queries].float().to(device).contiguous()
        missing = torch.zeros((outfits.shape[0], S), dtype=torch.bool, device=device)
        missing[:, slots] = True
        if args.beam is None:
            err, ids = comp.complete(outfits, missing)
        else:
            err, ids = comp.complete_beam(outfits, missing, args.beam)
        if rank == 0:
            res = {"mode": "complete", "missing": slots, "depth": args.complete_depth, "metric": args.metric, "k": args.k,
                   "ids": ids.cpu().tolist(), "errors": err.cpu().tolist()}
            if args.beam is not None:
                res["beam"] = args.beam
            print(json.dumps(res))
        raise SystemExit(0)
    if args.mode == "revise":
        S = len(cats)
        cat_dtype = torch.bfloat16 if args.catalog_dtype == "bf16" else torch.float32
        catalogs = [dataset.data_per_category[s][lo:lo + n_local].to(device).to(cat_dtype).contiguous() for s in range(S)]
        comp = OutfitCompleter(model, catalogs, E, depth=args.complete_depth, k=args.k, metric=args.metric,
                               inv_scale=1.0 / dataset.scale, row_offsets=[lo] * S)
        outfits = dataset.data[:args.queries].float().to(device).contiguous()
        Q = outfits.shape[0]
        exclude = (torch.arange(Q, dtype=torch.int64, device=device).view(Q, 1, 1).expand(Q, S, 1)
                   if args.exclude_own_item else None)
        base, err, slot, ids = comp.revise(outfits, exclude=exclude)
        if rank == 0:
            print(json.dumps({"mode": "revise", "depth": args.complete_depth, "metric": args.metric, "k": args.k,
                              "base": base.cpu().tolist(), "errors": err.cpu().tolist(), "slots": slot.cpu().tolist(),
                              "ids": ids.cpu().tolist()}))
        raise SystemExit(0)
    shard = dataset.data_per_category[args.slot][lo:lo + n_local].to(device)
    if args.catalog_dtype == "bf16":
        shard = shard.to(torch.bfloat16)
    outfits = dataset.data[:args.queries].to(device)
    allowed = local_allowed(args.allowed_rows, lo, n_local, device)
    own = torch.arange(outfits.shape[0], dtype=torch.int64, device=device).view(-1, 1) if args.exclude_own_item else None
    if args.mode == "swap":
        if args.metric != "sqerr":
            raise Exception("Swap mode scores by squared reconstruction error.")
        scorer = SwapScorer(model, shard.contiguous(), E, k=args.k, inv_scale=1.0 / dataset.scale, row_offset=lo, allowed=allowed)
        res = [scorer.topk(outfits[q], args.slot, None if own is None else own[q]) for q in range(outfits.shape[0])]
        if rank == 0:
            print(json.dumps({"slot": args.slot, "mode": "swap", "metric": "sqerr", "k": args.k,
                              "indices": [i.cpu().tolist() for _, i in res], "scores": [s.cpu().tolist() for s, _ in res]}))
        raise SystemExit(0)
    rerank = args.mode == "rerank"
    scorer = ComplementarityScorer(shard.contiguous(), E, metric=args.metric, k=args.rerank_depth if rerank else args.k,
                                   inv_scale=1.0 / dataset.scale, row_offset=lo, allowed=allowed)
    p = predict_slot(model, outfits, args.slot, E)
    # large query batches: one tensor-core pass over the catalog, results identical to the row sweep
    scores, idx = scorer.topk_batched(p, own) if p.shape[0] >= ComplementarityScorer.TC_MIN_Q else scorer.topk(p, own)
    if rerank:
        swap = SwapScorer(model, shard.contiguous(), E, k=args.k, inv_scale=1.0 / dataset.scale, row_offset=lo, allowed=allowed)
        scores, idx = swap.rerank(outfits.float().contiguous(), args.slot, idx.contiguous())
        if rank == 0:
            print(json.dumps({"slot": args.slot, "mode": "rerank", "depth": args.rerank_depth, "k": args.k,
                              "indices": idx.cpu().tolist(), "scores": scores.cpu().tolist()}))
        raise SystemExit(0)
    if rank == 0:
        print(json.dumps({"slot": args.slot, "metric": args.metric, "k": args.k,
                          "indices": idx.cpu().tolist(), "scores": scores.cpu().tolist()}))
