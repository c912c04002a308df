"""GPU tests of the filtered complementarity top-k (codae_score_topk_filtered, codae_score_topk_batched_filtered,
codae_swap_error_topk_filtered; ComplementarityScorer / SwapScorer with `allowed` and `exclude`): a filtered-out row must behave
exactly as if it were absent from the catalog, and the batched path must still return exactly what the sweep returns."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _catalog(n, E, bf16, seed, specials=False):
    torch.manual_seed(seed)
    cat = torch.randn(n, E).abs() * (torch.rand(n, E) < 0.7)
    if n > 10:
        cat[n // 2] = cat[3]                      # exact duplicate rows: ties resolve to the lower index
    if specials and n > 10:
        cat[n // 3, 5] = float("nan")
        cat[n // 4, 0] = float("inf")
    return cat.to(torch.bfloat16) if bf16 else cat


def _queries(cat, Q, E, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(Q, E, generator=g).abs() * 0.3
    if cat.shape[0] > 10:
        q[0] = cat[3].float() * 0.5 + 0.01
    return q


def topk_filtered(scores, k, metric, row_offset, allowed=None, exclude=()):
    """fp64 restatement of the filtered top-k of one query: the best k (score, global index) pairs over the rows that are
    allowed (bool [n] or None) and not excluded (global indices; < 0 is padding), ties -> lower index, NaN never ranks."""
    s = scores.double()
    n = len(s)
    keep = torch.ones(n, dtype=torch.bool) if allowed is None else allowed.clone().bool()
    keep &= ~torch.isnan(s)
    for g in exclude:
        if 0 <= int(g) - row_offset < n:
            keep[int(g) - row_offset] = False
    rows = torch.nonzero(keep).flatten()
    key = s[rows] if metric == "sqerr" else -s[rows]
    order = np.lexsort((rows.numpy(), key.numpy()))[:k]
    return scores[rows[order]], rows[order] + row_offset


def _mask(n, density, k, seed):
    g = torch.Generator().manual_seed(seed)
    if density == "k-1":                          # exactly k - 1 eligible rows
        m = torch.zeros(n, dtype=torch.bool)
        m[torch.randperm(n, generator=g)[:max(k - 1, 0)]] = True
        return m
    return torch.rand(n, generator=g) < density


def _compacted(cat, E, q, metric, k, allow, inv_scale, row_offset):
    """Unfiltered sweep on catalog[allow], indices mapped back to the global rows of the full catalog."""
    from codae.tool.inference import ComplementarityScorer
    nz = torch.nonzero(allow).flatten()
    Q = q.shape[0]
    if len(nz) == 0:
        worst = float("inf") if metric == "sqerr" else float("-inf")
        return torch.full((Q, k), worst), torch.full((Q, k), -1, dtype=torch.int64)
    sc = ComplementarityScorer(cat[nz].to(DEV).contiguous(), E, metric=metric, k=k, inv_scale=inv_scale)
    s, i = (t.cpu() for t in sc.topk_local(q.to(DEV)))
    gi = torch.where(i >= 0, nz[i.clamp_min(0)] + row_offset, i)
    return s, gi


def _bits_equal(s, s_ref):
    return torch.equal(s.cpu().view(torch.int32), s_ref.cpu().view(torch.int32))


SWEEP = [  # n, E, Q, k, metric, bf16, density, specials
    (7, 16, 1, 10, "sqerr", False, 0.5, False), (7, 512, 5, 10, "cosine", True, 0.0, False),
    (5000, 16, 4, 10, "sqerr", True, 0.01, True), (5000, 512, 5, 64, "cosine", False, 0.5, True),
    (5000, 4096, 130, 10, "sqerr", False, "k-1", False), (5000, 512, 130, 128, "cosine", True, 1.0, False),
    (5000, 64, 4, 1, "sqerr", False, 0.5, True), (300_001, 512, 5, 10, "sqerr", True, 0.5, True),
    (300_001, 4096, 4, 64, "cosine", True, 0.01, False), (300_001, 16, 130, 128, "sqerr", False, "k-1", True),
    (300_001, 512, 1, 1, "cosine", False, 0.0, False), (300_001, 512, 5, 128, "cosine", False, 0.5, False),
]


@pytest.mark.parametrize("n,E,Q,k,metric,bf16,density,specials", SWEEP)
def test_sweep_filtered_equals_compacted_sweep(n, E, Q, k, metric, bf16, density, specials):
    from codae.tool.inference import ComplementarityScorer
    cat = _catalog(n, E, bf16, n + E + k, specials)
    q = _queries(cat, Q, E, Q + k)
    allow = _mask(n, density, k, n + Q)
    if n > 10 and density not in ("k-1", 0.0):
        allow[3] = allow[n // 2] = True           # the duplicate pair stays eligible
    sc = ComplementarityScorer(cat.to(DEV), E, metric=metric, k=k, inv_scale=0.5, row_offset=1000, allowed=allow.to(DEV))
    s, i = (t.cpu() for t in sc.topk_local(q.to(DEV)))
    s_ref, i_ref = _compacted(cat, E, q, metric, k, allow, 0.5, 1000)
    assert torch.equal(i, i_ref)
    assert _bits_equal(s, s_ref)
    if density == "k-1" and not specials:
        assert bool((i[:, :k - 1] >= 0).all()) and bool((i[:, k - 1:] == -1).all())


@pytest.mark.parametrize("bf16", [False, True])
def test_all_ones_mask_equals_unfiltered(bf16):
    from codae import _C
    n, E, Q, k = 20000, 256, 70, 10
    cat = _catalog(n, E, bf16, 5).to(DEV)
    q = _queries(cat.cpu(), Q, E, 6).to(DEV)
    ones = torch.ones(n, dtype=torch.uint8, device=DEV)
    no_ex = torch.empty((Q, 0), dtype=torch.int64, device=DEV)
    ws = _C.score_topk_workspace(DEV, Q, k)
    out = [(torch.empty(Q, k, device=DEV), torch.empty(Q, k, dtype=torch.int64, device=DEV)) for _ in range(2)]
    _C.score_topk(cat, E, 7, q, 0.5, _C.METRIC_SQERR, k, *out[0], ws)
    _C.score_topk(cat, E, 7, q, 0.5, _C.METRIC_SQERR, k, *out[1], ws, allow=ones, exclude=no_ex)
    assert torch.equal(out[0][1], out[1][1]) and _bits_equal(out[0][0], out[1][0])
    wsb = _C.score_topk_batched_workspace(cat, E, Q, k)
    cnt, unc = torch.zeros(1, dtype=torch.int32, device=DEV), torch.empty(Q, dtype=torch.int32, device=DEV)
    b = (torch.empty(Q, k, device=DEV), torch.empty(Q, k, dtype=torch.int64, device=DEV))
    _C.score_topk_batched(cat, E, 7, q, 0.5, _C.METRIC_SQERR, k, *b, cnt, unc, wsb, allow=ones, exclude=no_ex)
    assert int(cnt[0]) == 0
    assert torch.equal(b[1], out[0][1]) and _bits_equal(b[0], out[0][0])


@pytest.mark.parametrize("metric,bf16", [("sqerr", False), ("cosine", True)])
def test_per_query_exclusion_equals_compacted(metric, bf16):
    from codae.tool.inference import ComplementarityScorer
    n, E, Q, k, off = 5000, 128, 5, 10, 1000
    cat = _catalog(n, E, bf16, 21)
    q = _queries(cat, Q, E, 22)
    sc = ComplementarityScorer(cat.to(DEV), E, metric=metric, k=k, inv_scale=0.5, row_offset=off)
    s0, i0 = (t.cpu().clone() for t in sc.topk_local(q.to(DEV)))
    ex = torch.full((Q, 4), -1, dtype=torch.int64)
    ex[:, 0] = i0[:, 0]                            # its own unfiltered top-1
    ex[:, 2] = off + n + 17                        # outside the shard: never matches
    s, i = (t.cpu() for t in sc.topk_local(q.to(DEV), exclude=ex.to(DEV)))
    for qi in range(Q):
        allow = torch.ones(n, dtype=torch.bool)
        allow[int(i0[qi, 0]) - off] = False
        rs, ri = _compacted(cat, E, q[qi:qi + 1], metric, k, allow, 0.5, off)
        assert torch.equal(i[qi:qi + 1], ri) and _bits_equal(s[qi:qi + 1], rs)
        assert int(i0[qi, 0]) not in i[qi].tolist()
    if metric == "sqerr":
        assert int(i0[0, 0]) == off + 3 and int(i[0, 0]) == off + n // 2      # excluding row 3 promotes its duplicate


GRID = [  # n, E, Q, k, metric, bf16, specials (the grid of the unfiltered batched tests)
    (7, 16, 1, 10, "sqerr", False, False), (7, 64, 129, 1, "cosine", True, False),
    (5000, 16, 63, 10, "sqerr", True, True), (5000, 64, 128, 64, "cosine", False, True),
    (5000, 512, 1000, 10, "sqerr", False, False), (5000, 512, 129, 10, "cosine", True, False),
    (5000, 1536, 63, 1, "sqerr", True, False), (5000, 4096, 129, 64, "sqerr", False, False),
    (300_001, 512, 1000, 10, "sqerr", True, True), (300_001, 512, 128, 64, "cosine", True, True),
    (300_001, 64, 1000, 10, "cosine", False, False), (300_001, 1536, 129, 10, "sqerr", False, True),
    (300_001, 4096, 63, 1, "cosine", True, False), (300_001, 4096, 1, 10, "sqerr", True, False),
]


def _exclusions(i_unf, m, n, off, seed):
    """[Q, m]: the unfiltered top entries first, then random rows of the shard, one out-of-shard id, -1 padding."""
    Q = i_unf.shape[0]
    g = torch.Generator().manual_seed(seed)
    ex = torch.randint(off, off + n, (Q, m), generator=g)
    t = min(m, i_unf.shape[1])
    ex[:, :t] = i_unf[:, :t]
    if m >= 4:
        ex[:, -1] = -1
        ex[:, -2] = off + n + 5
    return ex


@pytest.mark.parametrize("m", [1, 64])
@pytest.mark.parametrize("n,E,Q,k,metric,bf16,specials", GRID)
def test_batched_filtered_equals_filtered_sweep(n, E, Q, k, metric, bf16, specials, m):
    from codae.tool.inference import ComplementarityScorer
    off = 1000
    cat = _catalog(n, E, bf16, n + E + k, specials)
    q = _queries(cat, Q, E, Q + k).to(DEV)
    allow = _mask(n, 0.5, k, n + m).to(DEV)
    sc = ComplementarityScorer(cat.to(DEV).contiguous(), E, metric=metric, k=k, inv_scale=0.5, row_offset=off, allowed=allow)
    unf = ComplementarityScorer(cat.to(DEV).contiguous(), E, metric=metric, k=k, inv_scale=0.5, row_offset=off)
    ex = _exclusions(unf.topk_local(q)[1].cpu(), m, n, off, Q + m).to(DEV)
    s_ref, i_ref = (t.clone() for t in sc.topk_local(q, exclude=ex))
    s, i = sc.topk_local_batched(q, exclude=ex)
    assert torch.equal(i, i_ref)
    assert _bits_equal(s, s_ref)
    if n > 1000 and not specials:
        assert sc.last_fallbacks == 0
    hit = (i.cpu()[:, :, None] == ex.cpu()[:, None, :]) & (i.cpu()[:, :, None] >= 0)
    assert not bool(hit.any())
    ok = i.cpu() >= 0
    assert bool(allow.cpu()[(i.cpu() - off).clamp_min(0)][ok].all())


def test_tie_heavy_query_with_exclusion_falls_back():
    """More than k' identical rows at the k-th place cannot be certified: those queries fall back to the filtered sweep, which
    must honour their exclusions."""
    from codae.tool.inference import ComplementarityScorer
    n, E, k, Q = 20000, 64, 10, 200
    kp = min(2 * k + 32, 128)
    torch.manual_seed(3)
    cat = torch.rand(n, E)
    q = torch.rand(Q, E)
    tied = [5, 77, 150]
    winners = {}
    row = 100
    for qi in tied:
        winners[qi] = row
        for j in range(k - 1):
            cat[row] = q[qi] + 1e-3 * (j + 1); row += 1
        for _ in range(kp + 8):
            cat[row] = q[qi] + 2e-2; row += 1
    ex = torch.full((Q, 2), -1, dtype=torch.int64)
    for qi in tied:
        ex[qi, 0] = winners[qi]                    # the clear winner of each tied query
    allow = torch.ones(n, dtype=torch.bool)
    allow[torch.randperm(n)[:2000]] = False
    for qi in tied:                                # keep the tie block itself eligible
        allow[winners[qi]:winners[qi] + k - 1 + kp + 8] = True
    sc = ComplementarityScorer(cat.to(DEV), E, "sqerr", k, allowed=allow.to(DEV))
    exd = ex.to(DEV)
    s_ref, i_ref = (t.clone() for t in sc.topk_local(q.to(DEV), exclude=exd))
    s, i = sc.topk_local_batched(q.to(DEV), exclude=exd)
    assert sc.last_fallbacks == len(tied)
    assert torch.equal(i, i_ref) and _bits_equal(s, s_ref)
    for qi in tied:
        assert winners[qi] not in i[qi].tolist() and winners[qi] + 1 == int(i[qi, 0])


@pytest.mark.parametrize("n,E,Q,k,metric,bf16", [(5000, 512, 130, 10, "sqerr", False), (5000, 64, 64, 7, "cosine", True),
                                                 (7, 512, 3, 10, "sqerr", False)])
def test_batched_filtered_matches_oracle(n, E, Q, k, metric, bf16):
    from oracle import codae_oracle as O
    from codae.tool.inference import ComplementarityScorer
    off = 1000
    cat = _catalog(n, E, bf16, n + E + k)
    q = _queries(cat, Q, E, Q + k)
    allow = _mask(n, 0.5, k, 4)
    ex = torch.full((Q, 3), -1, dtype=torch.int64)
    ex[:, 0] = off + torch.arange(Q) % n
    sc = ComplementarityScorer(cat.to(DEV), E, metric=metric, k=k, inv_scale=0.5, row_offset=off, allowed=allow.to(DEV))
    s, i = (t.cpu() for t in sc.topk_local_batched(q.to(DEV), exclude=ex.to(DEV)))
    for qi in range(0, Q, 13):
        scores = O.score_candidates(cat.float(), q[qi], metric, inv_scale=0.5)
        ws, wi = topk_filtered(scores, k, metric, off, allowed=allow, exclude=ex[qi].tolist())
        m = len(wi)
        assert i[qi, :m].tolist() == wi.tolist(), (qi, i[qi, :m], wi)
        assert torch.all(i[qi, m:] == -1)
        assert np.allclose(s[qi, :m].numpy(), ws.numpy(), rtol=2e-5, atol=1e-6)


@pytest.mark.parametrize("batched", [False, True])
def test_shards_merge_equals_unsharded(batched):
    from codae import _C
    from codae.tool.inference import ComplementarityScorer, shard_rows
    n, E, k, G, Q = 30011, 512, 10, 4, 300
    torch.manual_seed(0)
    cat = torch.randn(n, E).abs().to(DEV)
    q = torch.randn(Q, E).abs().to(DEV)
    allow = _mask(n, 0.5, k, 8).to(DEV)
    ex = torch.full((Q, 8), -1, dtype=torch.int64)
    ex[:, 0] = torch.arange(Q) * 97 % n            # global ids spread over all shards
    ex[:, 1] = torch.arange(Q) * 31 % n
    ex = ex.to(DEV)
    full = ComplementarityScorer(cat, E, "sqerr", k, allowed=allow)
    ref_s, ref_i = (t.clone() for t in full.topk_local(q, exclude=ex))
    ps, pi = [], []
    for r in range(G):
        lo, c = shard_rows(n, G, r)
        sc = ComplementarityScorer(cat[lo:lo + c], E, "sqerr", k, row_offset=lo, allowed=allow[lo:lo + c])
        s, i = sc.topk_local_batched(q, exclude=ex) if batched else sc.topk_local(q, exclude=ex)
        ps.append(s.clone()); pi.append(i.clone())
    ms, mi = torch.empty_like(ref_s), torch.empty_like(ref_i)
    _C.topk_merge(torch.stack(ps), torch.stack(pi), _C.METRIC_SQERR, ms, mi)
    assert torch.equal(mi, ref_i) and _bits_equal(ms, ref_s)


def _swap_model(S, E, z, nin, nout, dtype, seed):
    from codae.model import EmbeddingDenoisingAutoencoder
    torch.manual_seed(seed)
    model = EmbeddingDenoisingAutoencoder(S * E, z, E, nin, nout, False)
    for lin in model.linears():
        torch.nn.init.uniform_(lin.bias, -0.05, 0.05)
    W = [lin.weight.detach().clone() for lin in model.linears()]
    b = [lin.bias.detach().clone() for lin in model.linears()]
    model = model.to(DEV).set_compute_dtype(dtype)
    return model, W, b


@pytest.mark.parametrize("cat_bf16", [False, True])
def test_swap_filtered_equals_compacted(cat_bf16):
    """The disallowed rows straddle the chunk boundaries (1024, 2048).  Two references: (a) the unfiltered scorer on the same
    catalog with the filtered-out rows replaced by far-away rows -- the same chunks, so the same GEMM schedule: bit for bit;
    (b) the unfiltered scorer on the compacted catalog -- its chunks hold other rows, and the DAE GEMM's split-K factor follows
    a chunk's row count (test_gpu_inference.py), so the errors agree to rounding and the indices exactly."""
    from codae.tool.inference import SwapScorer
    n, S, E, slot, k, chunk, off = 3000, 4, 64, 2, 10, 1024, 100
    model, W, b = _swap_model(S, E, 96, 2, 2, "fp32", 41)
    torch.manual_seed(42)
    cat = torch.rand(n, E) * 2
    outfit = torch.rand(S * E)
    cat[1020:1030] = outfit[slot * E:(slot + 1) * E] * 2       # near-perfect swaps, all but one filtered out
    cat[2040:2056] = outfit[slot * E:(slot + 1) * E] * 2 + 1e-3
    allow = torch.rand(n) < 0.7
    allow[1000:1050] = False
    allow[2040:2070] = False
    allow[1025] = True
    ex = torch.tensor([off + 1025, -1, off + 5000], dtype=torch.int64)     # ... and that one excluded
    if cat_bf16:
        cat = cat.to(torch.bfloat16)
    keep = allow.clone()
    keep[1025] = False
    sc = SwapScorer(model, cat.to(DEV), E, k=k, inv_scale=0.5, row_offset=off, chunk=chunk, allowed=allow.to(DEV))
    s, i = (t.cpu() for t in sc.topk_local(outfit.to(DEV), slot, exclude=ex.to(DEV)))
    far = cat.clone()
    far[~keep] = 1e4
    s_a, i_a = (t.cpu() for t in SwapScorer(model, far.to(DEV), E, k=k, inv_scale=0.5, row_offset=off,
                                            chunk=chunk).topk_local(outfit.to(DEV), slot))
    assert torch.equal(i, i_a) and _bits_equal(s, s_a)
    nz = torch.nonzero(keep).flatten()
    s_b, i_b = (t.cpu() for t in SwapScorer(model, cat[nz].contiguous().to(DEV), E, k=k, inv_scale=0.5,
                                            chunk=chunk).topk_local(outfit.to(DEV), slot))
    assert torch.equal(i, nz[i_b] + off)
    assert np.allclose(s.numpy(), s_b.numpy(), rtol=1e-5, atol=1e-6)
    assert not any(1020 <= int(x) - off < 1030 or 2040 <= int(x) - off < 2056 for x in i)


def test_swap_filtered_matches_oracle():
    from oracle import codae_oracle as O
    from codae.tool.inference import SwapScorer
    n, S, E, slot, k, off = 700, 3, 64, 1, 8, 100
    model, W, b = _swap_model(S, E, 96, 2, 2, "fp32", 43)
    torch.manual_seed(44)
    cat = torch.rand(n, E) * 2
    outfit = torch.rand(S * E)
    allow = torch.rand(n) < 0.5
    sc = SwapScorer(model, cat.to(DEV), E, k=k, inv_scale=0.5, row_offset=off, chunk=256, allowed=allow.to(DEV))
    unf = SwapScorer(model, cat.to(DEV), E, k=k, inv_scale=0.5, row_offset=off, chunk=256)
    top = int(unf.topk_local(outfit.to(DEV), slot)[1][0])
    ex = torch.tensor([top, -1], dtype=torch.int64)
    s, i = (t.cpu() for t in sc.topk_local(outfit.to(DEV), slot, exclude=ex.to(DEV)))
    err = O.score_swaps(W, b, model.relu, outfit, slot, E, cat.float(), inv_scale=0.5)
    ws, wi = topk_filtered(err, k, "sqerr", off, allowed=allow, exclude=[top])
    assert i.tolist() == wi.tolist()
    assert np.allclose(s.numpy(), ws.numpy(), rtol=1e-5, atol=1e-6)


def test_full_size_planted_near_copies_filtered():
    """10 M x 512 bf16, Q = 1024, k = 10, 50 % mask and own-item exclusion (query q never gets row q).  Near-copies of the
    queries planted on excluded and on disallowed rows never appear; those planted on eligible rows come back in order; the
    batched result equals the filtered sweep."""
    from codae.tool.inference import ComplementarityScorer
    n, E, k, Q = 10_000_000, 512, 10, 1024
    g = torch.Generator(device=DEV).manual_seed(12)
    cat = torch.rand((n, E), generator=g, device=DEV).to(torch.bfloat16)
    q = torch.rand((Q, E), generator=g, device=DEV)
    allow = torch.rand(n, generator=g, device=DEV) < 0.5
    allow[:Q] = True                                           # row q is eligible: only the exclusion removes it
    own = torch.arange(Q, dtype=torch.int64, device=DEV).view(Q, 1)
    banned, eligible = {}, {}
    for qi in (0, 17, 500, 1023):
        cat[qi] = q[qi].to(cat.dtype)                          # the best possible row, on the excluded row q
        off_rows = torch.nonzero(~allow[Q:Q + 100_000]).flatten()[qi * 3:qi * 3 + 3] + Q
        for j, r in enumerate(off_rows.tolist()):
            cat[r] = (q[qi] + 1e-2 * (j + 1)).to(cat.dtype)    # near-copies on disallowed rows
        on_rows = torch.nonzero(allow[Q + 100_000:]).flatten()[qi * 20:qi * 20 + k] + Q + 100_000
        for j, r in enumerate(on_rows.tolist()):
            cat[r] = (q[qi] + 2e-2 * (j + 1)).to(cat.dtype)
        banned[qi] = [qi] + off_rows.tolist()
        eligible[qi] = on_rows.tolist()
    sc = ComplementarityScorer(cat, E, "sqerr", k, allowed=allow)
    s, i = (t.clone() for t in sc.topk_local_batched(q, exclude=own))
    assert sc.last_fallbacks == 0
    for qi in banned:
        assert not set(banned[qi]) & set(i[qi].tolist())
        assert i[qi].tolist() == eligible[qi]
    assert not bool((i == own).any())
    assert bool(allow[i.flatten()].all())
    s_ref, i_ref = sc.topk_local(q, exclude=own)
    assert torch.equal(i, i_ref) and _bits_equal(s, s_ref)


def _guarded(bufs, nbytes, guard=4096):            # 0xff bytes: NaN as float32, -1 as integers
    buf = torch.full((guard + nbytes + guard,), 255, dtype=torch.uint8, device=DEV)
    bufs.append(buf)
    return buf[guard:guard + nbytes]


@pytest.mark.parametrize("batched", [False, True])
def test_filtered_outputs_stay_in_bounds(batched):
    from codae import _C
    n, E, Q, k, guard = 9000, 64, 200, 10, 4096
    torch.manual_seed(1)
    cat = torch.rand(n, E, device=DEV)
    q = torch.rand(Q, E, device=DEV)
    bufs = []
    allow = _guarded(bufs, n)
    allow.copy_((torch.rand(n, device=DEV) < 0.5).to(torch.uint8))
    ex = _guarded(bufs, Q * 256 * 8).view(torch.int64).view(Q, 256)
    ex.copy_(torch.randint(0, n, (Q, 256), device=DEV))
    s = _guarded(bufs, Q * k * 4).view(torch.float32).view(Q, k)
    i = _guarded(bufs, Q * k * 8).view(torch.int64).view(Q, k)
    if batched:
        ws = _guarded(bufs, _C.score_topk_batched_workspace(cat, E, Q, k).numel())
        cnt = _guarded(bufs, 4).view(torch.int32)
        unc = _guarded(bufs, Q * 4).view(torch.int32)
    else:
        ws = _guarded(bufs, _C.score_topk_workspace(DEV, Q, k).numel())
    before = [b.clone() for b in bufs]
    if batched:
        _C.score_topk_batched(cat, E, 0, q, 1.0, _C.METRIC_SQERR, k, s, i, cnt, unc, ws, allow=allow, exclude=ex)
    else:
        _C.score_topk(cat, E, 0, q, 1.0, _C.METRIC_SQERR, k, s, i, ws, allow=allow, exclude=ex)
    torch.cuda.synchronize()
    for b, b0 in zip(bufs, before):
        assert torch.equal(b[:guard], b0[:guard]) and torch.equal(b[-guard:], b0[-guard:])
    assert torch.equal(allow, before[0][guard:-guard]) and torch.equal(ex.flatten().view(torch.uint8), before[1][guard:-guard])
    if batched:
        assert int(cnt[0]) == 0
    assert not torch.isnan(s).any()
    assert bool(allow[i.flatten()].bool().all())
    assert not bool((i[:, :, None] == ex[:, None, :]).any())


def test_bad_filters_are_rejected():
    from codae import _C
    from codae.tool.inference import ComplementarityScorer, SwapScorer
    n, E, Q, k = 100, 64, 4, 5
    cat = torch.rand(n, E, device=DEV)
    q = torch.rand(Q, E, device=DEV)
    c, L = _C.ctx(DEV), _C.lib()
    ws = _C.score_topk_workspace(DEV, Q, k)
    s, i = torch.empty(Q, k, device=DEV), torch.empty(Q, k, dtype=torch.int64, device=DEV)
    ex = torch.zeros(Q, 300, dtype=torch.int64, device=DEV)
    P = _C.p

    def call(allow, exp, m, row_offset=0):
        return L.codae_score_topk_filtered(c, P(cat), _C.F32, n, E, E, row_offset, P(q), Q, 1.0, _C.METRIC_SQERR, k, allow, exp, m,
                                           P(s), P(i), P(ws), ws.numel(), _C.stream())
    assert call(None, P(ex), 257) == _C.EINVAL
    assert call(None, P(ex), -1) == _C.EINVAL
    assert call(None, P(ex), 0) == _C.EINVAL                    # a list pointer with n_exclude == 0
    assert call(None, None, 3) == _C.EINVAL
    assert call(None, P(ex), 3, row_offset=-1) == _C.EINVAL
    assert call(None, P(ex), 256) == _C.OK and call(None, None, 0) == _C.OK
    cnt, unc = torch.zeros(1, dtype=torch.int32, device=DEV), torch.empty(Q, dtype=torch.int32, device=DEV)
    wsb = _C.score_topk_batched_workspace(cat, E, Q, k)
    assert L.codae_score_topk_batched_filtered(c, P(cat), _C.F32, n, E, E, 0, P(q), Q, 1.0, _C.METRIC_SQERR, k, None, P(ex), 257,
                                               P(s), P(i), P(cnt), P(unc), P(wsb), wsb.numel(), _C.stream()) == _C.EINVAL
    y = torch.zeros(n, 2 * E, device=DEV)
    outfit = torch.zeros(2 * E, device=DEV)
    ws1 = _C.score_topk_workspace(DEV, 1, k)
    assert L.codae_swap_error_topk_filtered(c, P(outfit), P(cat), _C.F32, E, 0, n, E, 0, 2 * E, 1.0, P(y), 2 * E, 0, k, None,
                                            P(ex), 0, P(s), P(i), P(ws1), ws1.numel(), _C.stream()) == _C.EINVAL
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="bool or uint8"):
        ComplementarityScorer(cat, E, k=k, allowed=torch.ones(n, dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError, match="shape"):
        ComplementarityScorer(cat, E, k=k, allowed=torch.ones(n + 1, dtype=torch.bool, device=DEV))
    with pytest.raises(RuntimeError, match="device"):
        ComplementarityScorer(cat, E, k=k, allowed=torch.ones(n, dtype=torch.bool))
    sc = ComplementarityScorer(cat, E, k=k)
    with pytest.raises(RuntimeError, match="int64"):
        sc.topk_local(q, exclude=torch.zeros(Q, 1, dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError, match="shape"):
        sc.topk_local(q, exclude=torch.zeros(Q + 1, 1, dtype=torch.int64, device=DEV))
    with pytest.raises(RuntimeError, match="shape"):
        sc.topk_local_batched(q, exclude=torch.zeros(Q, 257, dtype=torch.int64, device=DEV))
    with pytest.raises(RuntimeError, match="device"):
        sc.topk(q, exclude=torch.zeros(Q, 1, dtype=torch.int64))
    model, _, _ = _swap_model(2, E, 32, 2, 2, "fp32", 1)
    sw = SwapScorer(model, cat, E, k=k)
    with pytest.raises(RuntimeError, match="shape"):
        sw.topk_local(outfit, 0, exclude=torch.zeros(1, 2, dtype=torch.int64, device=DEV))


@pytest.mark.parametrize("mode", ["slot", "swap"])
def test_script_filter_flags(tmp_path, mode):
    n = 3000
    allowed = np.arange(0, n, 3, dtype=np.int64)
    allowed = np.concatenate([allowed, np.arange(4)])           # the queries' own rows are allowed: only the exclusion drops them
    path = os.path.join(str(tmp_path), "allowed.npy")
    np.save(path, allowed)
    args = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config",
            os.path.join(PKG, "config", "embedding.yaml"), "--synthetic", str(n), "--slot", "1", "--k", "6", "--queries", "4",
            "--mode", mode, "--exclude_own_item", "--allowed_rows", path]
    r = subprocess.run([sys.executable] + args, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    ok = set(allowed.tolist())
    assert len(res["indices"]) == 4
    for q, row in enumerate(res["indices"]):
        assert len(row) == 6 and q not in row
        assert all(i in ok for i in row)
