"""Outfit compatibility scoring (CompatibilityScorer.score_local) against what a user writes without it: S predict_slot calls (the
autograd forward of the model, one per hidden slot) and the leave-one-out errors, score and odd slot computed in torch.  One JSON
line per case.

Cases: embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)) with the bf16 and the fp32-parity engines at Q = 128,
10 000 and 100 000 outfits; the polyvore-shaped model (8 slots x 512, 10 x Linear(4096, 4096)) in bf16 at Q = 10 000.  The two
paths alternate in one process after a warm-up of both, timed with CUDA events around whole calls.  Their outputs are compared in
the same run: the largest relative slot-error difference and the odd slots that differ where the top two errors are not a
near-tie (within the engine's tolerance).  The card's name and power limit are read in the same run.

    python tools/bench_outfit_compat.py [--reps 3] [--out profiles/r06_outfit_compat.jsonl]
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


def baseline(model, outfits, S, E, block):
    """S predict_slot calls per block of outfits (the autograd path at the same row count as one scorer chunk), then the errors,
    their slot-order sum and the argmax in torch."""
    from codae.tool.inference import predict_slot
    errs = []
    for c0 in range(0, outfits.shape[0], block):
        x = outfits[c0:c0 + block]
        cols = [((predict_slot(model, x, s, E) - x[:, s * E:(s + 1) * E]) ** 2).sum(1) for s in range(S)]
        errs.append(torch.stack(cols, 1))
    err = torch.cat(errs)
    score = err[:, 0].clone()
    for s in range(1, S):
        score += err[:, s]
    return err, score, err.argmax(1)


def compare(e0, o0, e1, o1, rtol):
    """(largest relative slot-error difference, odd slots that differ where the top two errors are further apart than the
    engine's tolerance)."""
    e0, e1 = e0.double().cpu(), e1.double().cpu()
    rel = ((e0 - e1).abs() / e0.abs().clamp_min(1e-30)).max().item()
    top2 = e0.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 4 * rtol * top2[:, 0]
    return rel, int(((o0.cpu() != o1.cpu()) & clear).sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", type=str, default=None, help="also append the lines to this file")
    args = ap.parse_args()
    from codae.tool.inference import CompatibilityScorer
    dev = torch.device("cuda", 0)
    name = card()
    E = 512
    g = torch.Generator(device=dev).manual_seed(0)
    out = open(args.out, "a") if args.out else None
    cases = [("embedding", 3, 1536, "bf16", 128), ("embedding", 3, 1536, "bf16", 10_000), ("embedding", 3, 1536, "bf16", 100_000),
             ("embedding", 3, 1536, "fp32", 128), ("embedding", 3, 1536, "fp32", 10_000), ("embedding", 3, 1536, "fp32", 100_000),
             ("polyvore", 8, 4096, "bf16", 10_000)]
    for shape, S, z, engine, Q in cases:
        model = model_for(S, E, z, engine, dev)
        outfits = torch.rand((Q, S * E), generator=g, device=dev)
        sc = CompatibilityScorer(model, E)
        block = sc.chunk_outfits

        def ours():
            return sc.score_local(outfits)

        def theirs():
            return baseline(model, outfits, S, E, block)
        c_e, c_s, c_o = (t.clone() for t in ours())
        b_e, b_s, b_o = theirs()                           # warm-up of both at this shape
        t_c, t_b = [], []
        for _ in range(args.reps):
            t_c.append(timed(ours))
            t_b.append(timed(theirs))
        rel, far = compare(b_e, b_o, c_e, c_o, RTOL[engine])
        line = {"model": "%s (io %d, 10 x %d^2)" % (shape, S * E, z), "engine": engine, "Q": Q, "slots": S,
                "chunk_outfits": block, "ms_scorer_min": round(min(t_c), 3), "ms_predict_slot_loop_min": round(min(t_b), 3),
                "ms_scorer_median": round(statistics.median(t_c), 3),
                "ms_predict_slot_loop_median": round(statistics.median(t_b), 3),
                "loop_over_scorer": round(min(t_b) / min(t_c), 3),
                "M_rows_per_s_scorer": round(Q * S / min(t_c) / 1e3, 3), "M_rows_per_s_loop": round(Q * S / min(t_b) / 1e3, 3),
                "max_rel_slot_err_diff": rel, "odd_differing_beyond_near_tie": far, "reps": args.reps, "card": name}
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()
        del sc, model, outfits
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
