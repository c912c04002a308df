"""GPU tests of outfit revision (codae_revise_build / codae_revise_error; OutfitCompleter.revise_candidates / revise_local / revise;
4_complementarity_inference.py --mode revise).  Every outfit is scored as given and with each candidate of each slot swapped in; the
swaps below the outfit's own error are ranked.  A GEMM row depends only on that row and on the launch's 128-row tile count, so at
chunks of <= 128 rows a swap's error is what SwapScorer.rerank and complete give for the same outfit row, bit for bit."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG
from test_gpu_outfit_complete import _bits_equal, _catalogs, _guarded, _model

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ENGINES = ["fp32", "fp32_simt", "bf16"]
RTOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-2}
CAT_DTYPES = [torch.float32, torch.bfloat16]


def _listed(res, q):
    """[(error, slot, id)] of outfit q's listed swaps."""
    _, err, slot, ids = (t.cpu() for t in res)
    n = int(torch.isfinite(err[q]).sum())
    assert bool(torch.isinf(err[q, n:]).all()) and bool((slot[q, n:] == -1).all()) and bool((ids[q, n:] == -1).all()), q
    return [(float(err[q, e]), int(slot[q, e]), int(ids[q, e])) for e in range(n)]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_one_open_slot_is_rerank_below_base(engine, cat_dtype):
    """keep leaves only slot s open: the listed swaps are SwapScorer.rerank_local's entries below the base error, in the same order,
    errors and ids bit for bit; the base is complete_local's error of the outfit with nothing missing."""
    from codae.tool import OutfitCompleter, SwapScorer
    S, E, Q, depth = 3, 64, 40, 8
    model, _, _ = _model(S, E, engine, 201)
    g = torch.Generator(device=DEV).manual_seed(202)
    cats = _catalogs(S, E, [300, 300, 300], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    cand = torch.randint(0, 300, (Q, S, depth), generator=g, device=DEV)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=depth, inv_scale=0.7, chunk=128)
    none = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    e0, _ = comp.complete_local(outfits, none, cand)
    for s in range(S):
        keep = torch.ones((Q, S), dtype=torch.bool, device=DEV)
        keep[:, s] = False
        res = [t.clone() for t in comp.revise(outfits, keep=keep, candidates=cand)]
        assert _bits_equal(res[0], e0[:, 0])
        ws, wi = SwapScorer(model, cats[s], E, k=depth, inv_scale=0.7, chunk=128).rerank_local(outfits, s, cand[:, s].contiguous())
        ws, wi, base = ws.cpu(), wi.cpu(), res[0].cpu()
        n_any = 0
        for q in range(Q):
            want = [(float(ws[q, e]), s, int(wi[q, e])) for e in range(depth) if float(ws[q, e]) < float(base[q])]
            got = _listed(res, q)
            assert got == want, (s, q, got, want)
            n_any += len(got)
        assert n_any > 0, s


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_fed_back_swaps_give_complete_errors(engine, cat_dtype):
    """Each returned (slot, id), fed to complete_local as that slot missing with [id] as its list, gives the same error bit for bit."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 4, 32, 30, 6
    model, _, _ = _model(S, E, engine, 211)
    g = torch.Generator(device=DEV).manual_seed(212)
    cats = _catalogs(S, E, [200] * S, cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=10, inv_scale=0.5, chunk=100)
    base, err, slot, ids = (t.clone() for t in comp.revise(outfits))
    rows = [(q, e) for q in range(Q) for e in range(10) if int(slot[q, e]) >= 0]
    assert len(rows) > Q
    qs = torch.tensor([q for q, _ in rows], device=DEV)
    es = torch.tensor([e for _, e in rows], device=DEV)
    missing = torch.zeros((len(rows), S), dtype=torch.bool, device=DEV)
    missing[torch.arange(len(rows), device=DEV), slot[qs, es]] = True
    one = torch.full((len(rows), S, 1), -1, dtype=torch.int64, device=DEV)
    one[torch.arange(len(rows), device=DEV), slot[qs, es], 0] = ids[qs, es]
    fb = OutfitCompleter(model, cats, E, depth=1, k=1, inv_scale=0.5, chunk=100)
    got, gid = fb.complete_local(outfits[qs], missing, one)
    assert _bits_equal(got[:, 0], err[qs, es]) and torch.equal(gid[:, 0].max(1).values, ids[qs, es])
    assert bool((err[qs, es] < base[qs]).all())


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("S,Q", [(3, 40), (2, 64)])
def test_stage_one_is_predict_slot_topk(engine, S, Q):
    """Q S <= 128: revise_candidates is a per-slot ComplementarityScorer.topk on predict_slot's reconstruction with the same
    exclusions, ids bit for bit; Q = 64 open outfits per slot take the topk_batched branch, fewer the row sweep."""
    from codae.tool import ComplementarityScorer, OutfitCompleter
    from codae.tool.inference import predict_slot
    E, depth = 64, 6
    model, _, _ = _model(S, E, engine, 221 + S)
    g = torch.Generator(device=DEV).manual_seed(222)
    cats = _catalogs(S, E, [700] * S, torch.float32, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    exclude = torch.randint(-1, 700, (Q, S, 5), generator=g, device=DEV)
    for metric in ("sqerr", "cosine"):
        comp = OutfitCompleter(model, cats, E, depth=depth, metric=metric, inv_scale=0.5)
        for keep in (None, torch.rand((Q, S), generator=g, device=DEV) < 0.3):
            cand = comp.revise_candidates(outfits, keep, exclude)
            for s in range(S):
                rows = torch.arange(Q, device=DEV) if keep is None else torch.nonzero(~keep[:, s]).view(-1)
                sc = ComplementarityScorer(cats[s], E, metric=metric, k=depth, inv_scale=0.5)
                y = predict_slot(model, outfits, s, E)[rows]
                ex = exclude[rows, s].contiguous()
                _, want = sc.topk_batched(y, ex) if rows.numel() >= ComplementarityScorer.TC_MIN_Q else sc.topk(y, ex)
                assert torch.equal(cand[rows, s], want), (metric, s)
                if keep is not None:
                    assert bool((cand[keep[:, s], s] == -1).all())


def _oracle(W, b, relu, outfits, cand, cats, inv_scale):
    """fp64 brute force: per outfit (base error, sorted [(error, s depth + c, slot, id)] of every swap whose row exists)."""
    Q, S, depth = cand.shape
    E = outfits.shape[1] // S
    Wd = [w.to(DEV).double() for w in W]
    bd = [v.to(DEV).double() for v in b]

    def errs(x):
        h = x.double()
        for w, v, rl in zip(Wd, bd, relu):
            h = h @ w.T + v
            if rl:
                h = torch.relu(h)
        return ((h - x.double()) ** 2).sum(1).cpu().tolist()
    out = []
    for q in range(Q):
        rows, meta = [outfits[q].clone()], []
        for s in range(S):
            for c in range(depth):
                i = int(cand[q, s, c])
                if 0 <= i < cats[s].shape[0]:
                    x = outfits[q].clone()
                    x[s * E:(s + 1) * E] = cats[s][i, :E].float() * inv_scale
                    rows.append(x)
                    meta.append((s * depth + c, s, i))
        e = errs(torch.stack(rows))
        out.append((e[0], sorted((e[n + 1], key, s, i) for n, (key, s, i) in enumerate(meta))))
    return out


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_matches_fp64_oracle(engine, cat_dtype):
    """Caller-supplied lists with padding (-1) and ids outside the catalogs, a slot listing nothing: the base, the listed errors and
    ids agree with an fp64 brute force over every (outfit, slot, candidate), ids except at near-ties."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth, k = 4, 32, 24, 5, 12
    model, W, b = _model(S, E, engine, 231)
    rtol = RTOL[engine]
    g = torch.Generator(device=DEV).manual_seed(232)
    cats = _catalogs(S, E, [30 + 7 * s for s in range(S)], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    cand = torch.randint(-1, 45, (Q, S, depth), generator=g, device=DEV)
    cand[3, 1] = -1
    comp = OutfitCompleter(model, cats, E, depth=depth, k=k, inv_scale=0.5, chunk=250)
    res = [t.clone() for t in comp.revise_local(outfits, cand)]
    ref = _oracle(W, b, model.relu, outfits, cand.cpu(), cats, 0.5)
    tol = lambda v: 4 * rtol * abs(v) + 1e-6
    n_listed = 0
    for q, (base, swaps) in enumerate(ref):
        assert abs(float(res[0][q]) - base) <= rtol * abs(base) + 1e-6, q
        got = _listed(res, q)
        below = [t for t in swaps if t[0] < base]
        n_sure = len([t for t in below if base - t[0] > tol(base)])
        assert min(k, n_sure) <= len(got) <= min(k, len(below) + len([t for t in swaps if abs(t[0] - base) <= tol(base)])), q
        allv = [t[0] for t in swaps]
        for e, (ge, gs, gi) in enumerate(got):
            np.testing.assert_allclose(ge, allv[e], rtol=rtol, atol=1e-6)
            lo = allv[e - 1] if e else -np.inf
            hi = allv[e + 1] if e + 1 < len(allv) else np.inf
            if allv[e] - lo > tol(allv[e]) and hi - allv[e] > tol(allv[e]):
                assert (gs, gi) == swaps[e][2:], (q, e, (gs, gi), swaps[e])
        assert all(s != 1 for _, s, _ in got) or q != 3
        n_listed += len(got)
    assert n_listed > Q


@pytest.mark.parametrize("engine", ENGINES)
def test_independent_of_other_outfits_and_repeatable(engine):
    """13 grid rows per outfit, chunk 130 = 10 outfits: the other outfits of the target's chunk are replaced, then the chunk is
    permuted; the target's results stay bit-identical, and two runs agree."""
    from codae.tool import OutfitCompleter
    S, E, Q, t, depth = 3, 64, 20, 4, 4
    model, _, _ = _model(S, E, engine, 241)
    g = torch.Generator(device=DEV).manual_seed(242)
    cats = _catalogs(S, E, [50, 50, 50], torch.float32, g)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=6, chunk=130)
    a = torch.rand((Q, S * E), generator=g, device=DEV)
    ca = torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    ra = [x.clone() for x in comp.revise_local(a, ca)]
    rb = comp.revise_local(a, ca)
    assert all(_bits_equal(x, y) for x, y in zip(ra, rb))
    b, cb = torch.rand((Q, S * E), generator=g, device=DEV), torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    b[t], cb[t] = a[t], ca[t]
    rc = comp.revise_local(b, cb)
    assert all(_bits_equal(x[t], y[t]) for x, y in zip(ra, rc))
    perm = torch.randperm(10, generator=torch.Generator().manual_seed(9))
    perm = perm[perm != t]
    perm = torch.cat([perm[:6], torch.tensor([t]), perm[6:]]).to(DEV)
    c, cc = a.clone(), ca.clone()
    c[:10], cc[:10] = a[perm], ca[perm]
    rd = comp.revise_local(c, cc)
    assert all(_bits_equal(x[t], y[6]) for x, y in zip(ra, rd))
    assert all(_bits_equal(x[10:], y[10:]) for x, y in zip(ra, rd))


@pytest.mark.parametrize("engine", ENGINES)
def test_edge_cases(engine):
    """keep everything: a base and no swaps.  A NaN in an outfit: NaN base, no swaps, the other outfits bit-identical.  A NaN
    candidate row never lists.  The held item proposed again (x' equal to the outfit) never lists."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 3, 64, 12, 4
    model, _, _ = _model(S, E, engine, 251)
    g = torch.Generator(device=DEV).manual_seed(252)
    cats = _catalogs(S, E, [40, 40, 40], torch.float32, g)
    outfits = torch.cat([cats[s][:Q] * 0.5 for s in range(S)], 1)          # outfit q holds row q of every catalog
    cand = torch.randint(0, 40, (Q, S, depth), generator=g, device=DEV)
    cand[:, :, 0] = torch.arange(Q, device=DEV).view(Q, 1)                   # the held item, first in every list
    comp = OutfitCompleter(model, cats, E, depth=depth, k=3 * depth, inv_scale=0.5, chunk=100)
    ra = [x.clone() for x in comp.revise_local(outfits, cand)]
    assert bool(torch.isfinite(ra[0]).all())
    for q in range(Q):
        assert all(i != q for _, _, i in _listed(ra, q)), q
    keep = torch.ones((Q, S), dtype=torch.bool, device=DEV)
    base, err, slot, ids = comp.revise(outfits, keep=keep, candidates=cand)
    assert _bits_equal(base, ra[0]) and bool(torch.isinf(err).all()) and bool((slot == -1).all()) and bool((ids == -1).all())
    x = outfits.clone()
    x[3, 1 * E + 5] = float("nan")
    res = [t.clone() for t in comp.revise_local(x, cand)]
    assert bool(torch.isnan(res[0][3])) and _listed(res, 3) == []
    other = torch.arange(Q, device=DEV) != 3
    assert all(_bits_equal(u[other], v[other]) for u, v in zip(res, ra))
    cats2 = [c.clone() for c in cats]
    cats2[2][7, 3] = float("nan")
    cand2 = cand.clone()
    cand2[:, 2, 1] = 7
    comp2 = OutfitCompleter(model, cats2, E, depth=depth, k=3 * depth, inv_scale=0.5, chunk=100)
    res = comp2.revise_local(outfits, cand2)
    for q in range(Q):
        assert all(not (s == 2 and i == 7) for _, s, i in _listed(res, q)), q


def _planted_model(S, E, engine):
    """Square layers, every Linear the identity but the last, which maps every slot to the mean of all slots: an outfit's error is
    zero exactly when its slots are equal.  Inputs are >= 0, so the ReLUs pass."""
    from codae.model import EmbeddingDenoisingAutoencoder
    io = S * E
    model = EmbeddingDenoisingAutoencoder(io, io, E, 2, 2, False)
    lins = model.linears()
    with torch.no_grad():
        for lin in lins:
            lin.weight.copy_(torch.eye(io))
            lin.bias.zero_()
        lins[-1].weight.copy_(torch.eye(E).repeat(S, S) / S)
    return model.to(DEV).set_compute_dtype(engine)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_planted_replacement(engine, cat_dtype):
    """Outfits hold copies of one item v in every slot but slot 3, which holds a random w; slot 3's catalog holds a copy of v.  Stage 1
    reads slot 3 as a multiple of v, so cosine finds the copy, and replacing w by it (error ~ 0) is the first swap.  Outfits whose
    slots are all v cannot improve: no swap lists."""
    from codae.tool import OutfitCompleter
    S, E, Q, n = 4, 32, 40, 300
    model = _planted_model(S, E, engine)
    g = torch.Generator(device=DEV).manual_seed(261)
    v = torch.rand((Q, E), generator=g, device=DEV).to(torch.bfloat16).float()
    w = torch.rand((Q, E), generator=g, device=DEV).to(torch.bfloat16).float()
    outfits = v.repeat(1, S)
    odd = torch.arange(Q, device=DEV) % 2 == 0
    outfits[odd, 3 * E:] = w[odd]
    cats, planted = [], None
    for s in range(S):
        cat = torch.rand((n, E), generator=g, device=DEV)
        if s == 3:
            planted = torch.randperm(n, generator=torch.Generator().manual_seed(5))[:Q].to(DEV)
            cat[planted] = v
        cats.append(cat.to(cat_dtype))
    comp = OutfitCompleter(model, cats, E, depth=4, k=3, metric="cosine")
    base, err, slot, ids = comp.revise(outfits)
    assert bool((base[odd] > 1e-2).all()) and bool((base[~odd] <= 1e-4).all())
    assert torch.equal(slot[odd, 0], torch.full_like(slot[odd, 0], 3)) and torch.equal(ids[odd, 0], planted[odd])
    assert bool((err[odd, 0] <= 1e-4).all())
    assert bool(torch.isinf(err[~odd]).all()) and bool((ids[~odd] == -1).all())


def test_kernel_contract():
    """Built rows and errors inside NaN-filled guarded allocations: rows b < B, columns < io and err[pos[b]] of valid rows are written,
    nothing else.  Bad device data (a position outside the grid, an unrevised slot, slot_base past the pool, pool_id < 0) gives a
    zero row and no error; a swap equal to the outfit gets no error.  CODAE_EINVAL for bad host arguments."""
    from codae import _C
    S, E, Q, depth, guard = 3, 64, 5, 4, 4096
    io, G = S * E, 1 + S * depth
    g = torch.Generator(device=DEV).manual_seed(271)
    outfits = torch.rand((Q, io), generator=g, device=DEV)
    pool = torch.rand((Q * 2 * depth, E), generator=g, device=DEV)
    pool_id = torch.arange(pool.shape[0], dtype=torch.int64, device=DEV) + 1000
    pool_id[9] = -1
    slot_base = torch.full((Q, S), -1, dtype=torch.int64, device=DEV)
    slot_base[:, 0] = torch.arange(Q, device=DEV) * 2 * depth
    slot_base[:, 2] = torch.arange(Q, device=DEV) * 2 * depth + depth
    slot_base[4, 2] = pool.shape[0] - 2                              # candidates 2.. of outfit 4, slot 2 lie past the pool
    pool[3 * 2 * depth + 2] = outfits[3, :E] * 2                     # outfit 3, slot 0, candidate 2: the held item (x 0.5)
    pos = torch.tensor([0, 1, 1 * G + 1 + 2 * depth + 1, 1 * G + 2, 2 * G + 1 + depth, 3 * G, 3 * G + 3, 4 * G + 1 + 2 * depth + 2,
                        4 * G + 1 + 2 * depth + 1, -1, Q * G, 2 * G + G - 1], dtype=torch.int64, device=DEV)
    valid = [True, True, True, False, False, True, True, False, True, False, False, True]      # 1 G + 2 takes pool row 9
    no_err = [False] * 6 + [True] + [False] * 5                      # 3 G + 3: x' equals the outfit
    B = pos.numel()
    ld_x = io + 64
    for xdt in (torch.float32, torch.bfloat16):
        bufs = []
        x = _guarded(bufs, B * ld_x * (4 if xdt == torch.float32 else 2)).view(xdt).view(B, ld_x)
        err = _guarded(bufs, Q * G * 4).view(torch.float32)
        before = [t.clone() for t in bufs]
        _C.revise_build(outfits, S, E, slot_base, pool, pool_id, depth, pos, 0.5, x)
        y = torch.rand((B, io), generator=g, device=DEV)
        _C.revise_error(outfits, S, E, slot_base, pool, pool_id, depth, pos, 0.5, y, err)
        torch.cuda.synchronize()
        for bb, b0 in zip(bufs, before):
            assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])
        assert bool(torch.isnan(x[:, io:].float()).all())
        wrote = torch.zeros(Q * G, dtype=torch.bool)
        for b_, (p, ok, ne) in enumerate(zip(pos.tolist(), valid, no_err)):
            row = x[b_, :io].float()
            if not ok:
                assert not bool(row.any()), b_
                continue
            q, col = divmod(p, G)
            want = outfits[q].clone()
            if col:
                s, c = divmod(col - 1, depth)
                want[s * E:(s + 1) * E] = pool[int(slot_base[q, s]) + c] * 0.5
            assert torch.equal(row, want.to(xdt).float()), b_
            if ne:
                assert torch.equal(want, outfits[q])
                continue
            wrote[p] = True
            e_ref = ((y[b_] - want) ** 2).sum()
            assert abs(float(err[p]) - float(e_ref)) <= 1e-5 * float(e_ref), b_
        assert bool(torch.isnan(err.cpu()[~wrote]).all())
    c, L, P, st = _C.ctx(DEV), _C.lib(), _C.p, _C.stream()
    x = torch.empty((B, io), device=DEV)
    err = torch.empty(Q * G, device=DEV)

    def call(fn, **kw):
        a = dict(o=P(outfits), ldo=io, Q=Q, S=S, E=E, sb=P(slot_base), pool=P(pool), ldp=E, R=pool.shape[0], pid=P(pool_id),
                 depth=depth, pos=P(pos), B=B, x=P(x), xdt=_C.F32, ldx=io, y=P(x), ldy=io, err=P(err))
        a.update(kw)
        head = (c, a["o"], a["ldo"], a["Q"], a["S"], a["E"], a["sb"], a["pool"], a["ldp"], a["R"], a["pid"], a["depth"], a["pos"],
                a["B"], 0.5)
        if fn == "build":
            return L.codae_revise_build(*head, a["x"], a["xdt"], a["ldx"], st)
        return L.codae_revise_error(*head, a["y"], a["ldy"], a["err"], st)
    for fn in ("build", "error"):
        assert call(fn) == _C.OK
        common = (dict(o=None), dict(sb=None), dict(pool=None), dict(pid=None), dict(pos=None), dict(Q=0), dict(S=0), dict(S=65),
                  dict(E=0), dict(B=0), dict(depth=0), dict(depth=129), dict(Q=2 ** 31 // (1 + S * 128) + 1, depth=128),
                  dict(R=0), dict(ldp=E - 1), dict(ldo=io - 1), dict(o=outfits.data_ptr() + 2), dict(sb=slot_base.data_ptr() + 4),
                  dict(pid=pool_id.data_ptr() + 4), dict(pos=pos.data_ptr() + 4), dict(pool=pool.data_ptr() + 2))
        extra = ((dict(x=None), dict(ldx=io - 1), dict(xdt=7), dict(x=x.data_ptr() + 1)) if fn == "build" else
                 (dict(y=None), dict(err=None), dict(ldy=io - 1), dict(err=err.data_ptr() + 2)))
        for kw in common + extra:
            assert call(fn, **kw) == _C.EINVAL, (fn, kw)
    torch.cuda.synchronize()


def test_limits_raise_before_any_launch():
    from codae.tool import OutfitCompleter
    S, E = 3, 64
    model, _, _ = _model(S, E, "bf16", 281)
    cats = [torch.rand((20, E), device=DEV), None, torch.rand((20, E), device=DEV)]
    comp = OutfitCompleter(model, cats, E, depth=4)
    o = torch.rand((4, S * E), device=DEV)
    for kw, match in ((dict(keep=torch.zeros((4, S), dtype=torch.int32, device=DEV)), "bool"),
                      (dict(keep=torch.zeros((4, S), dtype=torch.bool)), "device"),
                      (dict(exclude=torch.zeros((4, S, 257), dtype=torch.int64, device=DEV)), "exclude"),
                      (dict(exclude=torch.zeros((4, S, 2), dtype=torch.int64)), "device"),
                      (dict(candidates=torch.zeros((4, S, 129), dtype=torch.int64, device=DEV)), "candidates"),
                      (dict(candidates=torch.zeros((4, S, 2), dtype=torch.int64)), "device")):
        with pytest.raises(RuntimeError, match=match):
            comp.revise(o, **kw)
    for bad in (o.double(), o.cpu(), o[:, :-1]):
        with pytest.raises(RuntimeError):
            comp.revise(bad)
    big = OutfitCompleter(model, cats, E, depth=128)
    with pytest.raises(RuntimeError, match="2\\*\\*31"):
        big.revise_candidates(torch.zeros(((2 ** 31 - 1) // (1 + S * 128) + 1, S * E), device=DEV))
    # a slot without a catalog is never revised, whatever its list holds
    cand = torch.randint(0, 20, (4, S, 4), device=DEV)
    _, _, slot, _ = comp.revise_local(o, cand)
    assert bool((slot != 1).all())


def _script(tmp_path, *extra):
    args = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config", os.path.join(PKG, "config", "embedding.yaml"),
            "--synthetic", "3000", "--queries", "16", "--mode", "revise", "--complete_depth", "4", "--k", "5", "--dtype", "bf16",
            "--catalog_dtype", "bf16"] + list(extra)
    return subprocess.run([sys.executable] + args, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)


def test_script_revise_mode(tmp_path):
    for extra in ([], ["--exclude_own_item"]):
        r = _script(tmp_path, *extra)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        res = json.loads(r.stdout.strip().splitlines()[-1])
        assert res["mode"] == "revise" and len(res["base"]) == 16
        for key in ("errors", "slots", "ids"):
            assert len(res[key]) == 16 and all(len(x) == 5 for x in res[key])
        for q in range(16):
            errs = res["errors"][q]
            assert errs == sorted(errs) and all(e < res["base"][q] or e == float("inf") for e in errs)
            for e, s, i in zip(errs, res["slots"][q], res["ids"][q]):
                assert (s == -1) == (i == -1) == (e == float("inf"))
                if extra:
                    assert i != q
    r = _script(tmp_path, "--allowed_rows", "x.npy")
    assert r.returncode != 0 and "revise" in r.stderr


DIST = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool import OutfitCompleter
from codae.tool.inference import shard_rows
dist.init_process_group("nccl")
r, G = dist.get_rank(), dist.get_world_size()
torch.cuda.set_device(r)
dev = torch.device("cuda", r)
S, E, Q, N = 3, 64, 101, 500
torch.manual_seed(5)
model = EmbeddingDenoisingAutoencoder(S * E, 96, E, 2, 2, False).to(dev).set_compute_dtype("bf16")
gen = torch.Generator().manual_seed(6)
outfits = torch.rand((Q, S * E), generator=gen).to(dev)
full = [torch.rand((N, E), generator=gen).to(dev) for _ in range(S)]
keep = (torch.rand((Q, S), generator=gen) < 0.3).to(dev)
exclude = torch.randint(0, N, (Q, S, 2), generator=gen).to(dev)
lo, n = shard_rows(N, G, r)
comp = OutfitCompleter(model, [c[lo:lo + n] for c in full], E, depth=4, k=6, row_offsets=[lo] * S, chunk=300)
one = OutfitCompleter(model, full, E, depth=4, k=6, chunk=300, process_group=None)
cand = comp.revise_candidates(outfits, keep, exclude)
res = [t.clone() for t in comp.revise(outfits, keep, exclude, cand)]
assert [tuple(t.shape) for t in res] == [(Q,), (Q, 6), (Q, 6), (Q, 6)]
for q in range(G):
    a, m = shard_rows(Q, G, q)
    want = one.revise_local(outfits[a:a + m], torch.where(keep[a:a + m].unsqueeze(2), -1, cand[a:a + m]))
    assert all(torch.equal(w.view(torch.int32) if w.dtype == torch.float32 else w,
                           t[a:a + m].view(torch.int32) if t.dtype == torch.float32 else t[a:a + m]) for w, t in zip(want, res)), q
dist.barrier()
dist.destroy_process_group()
c1 = one.revise_candidates(outfits, keep, exclude)
assert torch.equal(c1, cand)
if r == 0:
    print("REVISE DIST OK")
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_revise_on_two_gpus(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "revise_dist.py"
    script.write_text(DIST)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), PKG]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "REVISE DIST OK" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
