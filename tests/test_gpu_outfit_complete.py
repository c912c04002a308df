"""GPU tests of outfit completion (codae_complete_build / codae_complete_error; predict_missing; OutfitCompleter.candidates /
complete_local / complete; 4_complementarity_inference.py --mode complete).  Every combination of candidates for the missing slots
of an outfit is the completed outfit going through the model's GEMM chain; with one missing slot the arithmetic is
SwapScorer.rerank's, and a GEMM row depends only on that row and on the launch's 128-row tile count."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ENGINES = ["fp32", "fp32_simt", "bf16"]
RTOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-2}
CAT_DTYPES = [torch.float32, torch.bfloat16]


def _model(S, E, dtype, seed, z=96, nin=2, nout=2):
    from codae.model import EmbeddingDenoisingAutoencoder
    torch.manual_seed(seed)
    model = EmbeddingDenoisingAutoencoder(S * E, z, E, nin, nout, False)
    for lin in model.linears():
        torch.nn.init.uniform_(lin.bias, -0.05, 0.05)
    W = [lin.weight.detach().clone() for lin in model.linears()]
    b = [lin.bias.detach().clone() for lin in model.linears()]
    return model.to(DEV).set_compute_dtype(dtype), W, b


def _bits_equal(a, b):
    a, b = a.cpu().contiguous(), b.cpu().contiguous()
    if a.dtype == torch.int64:
        return torch.equal(a, b)
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _oracle(W, b, relu, outfits, missing, cand, cats, offsets, inv_scale):
    """fp64 brute force: per outfit, [(error, combination index, ids [S])] of every combination whose rows all exist, where x' holds
    each candidate row * inv_scale (computed in fp32, as the kernels build it) and error = || DAE(x') - x' ||^2 over io."""
    Q, S = missing.shape
    E = outfits.shape[1] // S
    Wd = [w.to(DEV).double() for w in W]
    bd = [v.to(DEV).double() for v in b]
    out = []
    for q in range(Q):
        ms = [s for s in range(S) if missing[q, s]]
        depth = cand.shape[2]
        rows, meta = [], []
        for c in range(depth ** len(ms)):
            x = outfits[q].clone()
            ids = [-1] * S
            ok = True
            for j, s in enumerate(ms):
                i = int(cand[q, s, (c // depth ** j) % depth])
                r = i - offsets[s]
                if i < 0 or not 0 <= r < cats[s].shape[0]:
                    ok = False
                    break
                x[s * E:(s + 1) * E] = cats[s][r, :E].float() * inv_scale
                ids[s] = i
            if ok:
                rows.append(x)
                meta.append((c, ids))
        res = []
        if rows:
            x = torch.stack(rows).double()
            h = x
            for w, v, rl in zip(Wd, bd, relu):
                h = h @ w.T + v
                if rl:
                    h = torch.relu(h)
            e = ((h - x) ** 2).sum(1).cpu()
            res = sorted([(float(e[n]), c, ids) for n, (c, ids) in enumerate(meta)], key=lambda t: (t[0], t[1]))
        out.append(res)
    return out


def _check_against_oracle(err, ids, ref, k, rtol):
    err, ids = err.cpu(), ids.cpu()
    for q, res in enumerate(ref):
        n = min(k, len(res))
        want = np.array([r[0] for r in res[:n]])
        np.testing.assert_allclose(err[q, :n].double().numpy(), want, rtol=rtol, atol=1e-6)
        assert bool(torch.isinf(err[q, n:]).all()) and bool((ids[q, n:] == -1).all()), q
        allv = [r[0] for r in res]
        for e in range(n):
            lo = allv[e - 1] if e else -np.inf
            hi = allv[e + 1] if e + 1 < len(allv) else np.inf
            if allv[e] - lo > 4 * rtol * abs(allv[e]) + 1e-6 and hi - allv[e] > 4 * rtol * abs(allv[e]) + 1e-6:
                assert ids[q, e].tolist() == res[e][2], (q, e, ids[q, e].tolist(), res[e][2])


def _catalogs(S, E, sizes, dtype, g):
    return [torch.rand((n, E), generator=g, device=DEV).to(dtype) for n in sizes]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
@pytest.mark.parametrize("S,E,depth,k,chunk", [(3, 64, 4, 10, 250), (5, 32, 8, 8, 1000), (8, 32, 1, 3, 8192), (4, 64, 8, 600, 250)])
def test_matches_fp64_oracle(engine, cat_dtype, S, E, depth, k, chunk):
    """Caller-supplied candidates with padding (-1) and ids outside the catalogs; m_q from 0 to 3 in one call; k below, equal to and
    above an outfit's number of valid combinations."""
    from codae.tool import OutfitCompleter
    Q = 24
    model, W, b = _model(S, E, engine, 10 + S)
    g = torch.Generator(device=DEV).manual_seed(S * depth)
    cats = _catalogs(S, E, [30 + 7 * s for s in range(S)], cat_dtype, g)
    offsets = [0] * S
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool)
    for q in range(Q):
        missing[q, torch.randperm(S, generator=torch.Generator().manual_seed(q))[:q % 4]] = True
    missing = missing.to(DEV)
    cand = torch.randint(-1, 45, (Q, S, depth), generator=g, device=DEV)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=min(k, 128), inv_scale=0.5, chunk=chunk)
    err, ids = comp.complete_local(outfits, missing, cand)
    ref = _oracle(W, b, model.relu, outfits, missing.cpu(), cand.cpu(), cats, offsets, 0.5)
    _check_against_oracle(err, ids, ref, min(k, 128), RTOL[engine])
    assert bool((ids.cpu()[~missing.cpu().unsqueeze(1).expand(-1, ids.shape[1], -1)] == -1).all())
    e2, i2 = comp.complete(outfits, missing, cand)
    assert _bits_equal(err, e2) and _bits_equal(ids, i2)


@pytest.mark.parametrize("engine", ENGINES)
def test_stage_one_identities(engine):
    """predict_missing with one slot is predict_slot bit for bit; candidates() lists are ComplementarityScorer.topk's ids on
    predict_missing's slot columns, for the row sweep (Q < 64) and the tensor-core batched path (Q >= 64)."""
    from codae.tool import ComplementarityScorer, OutfitCompleter
    from codae.tool.inference import predict_missing, predict_slot
    S, E = 3, 64
    model, _, _ = _model(S, E, engine, 3)
    g = torch.Generator(device=DEV).manual_seed(4)
    cats = _catalogs(S, E, [500, 700, 300], torch.float32, g)
    for Q in (10, 100):
        outfits = torch.rand((Q, S * E), generator=g, device=DEV)
        for slot in range(S):
            one = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
            one[:, slot] = True
            y = predict_missing(model, outfits, one, E)
            assert _bits_equal(y[:, slot * E:(slot + 1) * E].contiguous(), predict_slot(model, outfits, slot, E))
        missing = torch.rand((Q, S), generator=g, device=DEV) < 0.5
        missing[:, 0] = True
        for metric in ("sqerr", "cosine"):
            comp = OutfitCompleter(model, cats, E, depth=6, metric=metric, inv_scale=0.5)
            cand = comp.candidates(outfits, missing)
            y = predict_missing(model, outfits, missing, E)
            for s in range(S):
                rows = torch.nonzero(missing[:, s]).view(-1)
                if rows.numel() == 0:
                    continue
                _, want = ComplementarityScorer(cats[s], E, metric=metric, k=6, inv_scale=0.5).topk(y[rows, s * E:(s + 1) * E])
                assert torch.equal(cand[rows, s], want), (Q, s, metric)
                assert bool((cand[~missing[:, s], s] == -1).all())


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_one_missing_slot_is_rerank_bit_for_bit(engine, cat_dtype):
    from codae.tool import OutfitCompleter, SwapScorer
    S, E, Q, depth, k = 3, 64, 300, 8, 5
    model, _, _ = _model(S, E, engine, 21)
    g = torch.Generator(device=DEV).manual_seed(22)
    cats = _catalogs(S, E, [400, 400, 400], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    for slot, chunk in ((1, 1000), (2, 250)):
        missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
        missing[:, slot] = True
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, inv_scale=0.7, chunk=chunk)
        cand = comp.candidates(outfits, missing)
        err, ids = comp.complete(outfits, missing, cand)
        ws, wi = SwapScorer(model, cats[slot], E, k=k, inv_scale=0.7, chunk=chunk).rerank(outfits, slot, cand[:, slot].contiguous())
        assert _bits_equal(err, ws) and torch.equal(ids[:, :, slot], wi)
        others = [s for s in range(S) if s != slot]
        assert bool((ids[:, :, others] == -1).all())


@pytest.mark.parametrize("engine", ENGINES)
def test_results_do_not_depend_on_the_rest_of_the_chunk(engine):
    """Two missing slots, depth 4: 16 combinations per outfit, chunk 160 = 10 outfits, Q = 20.  The other outfits of the target's
    chunk are replaced (outfits and candidates), then the chunk is permuted; the target's results stay bit-identical, and two runs
    agree."""
    from codae.tool import OutfitCompleter
    S, E, Q, t, depth = 3, 64, 20, 4, 4
    model, _, _ = _model(S, E, engine, 31)
    g = torch.Generator(device=DEV).manual_seed(32)
    cats = _catalogs(S, E, [50, 50, 50], torch.float32, g)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=6, chunk=160)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 1:] = True
    a = torch.rand((Q, S * E), generator=g, device=DEV)
    ca = torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    ra = [x.clone() for x in comp.complete_local(a, missing, ca)]
    rb = comp.complete_local(a, missing, ca)
    assert all(_bits_equal(x, y) for x, y in zip(ra, rb))
    b, cb = torch.rand((Q, S * E), generator=g, device=DEV), torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    b[t], cb[t] = a[t], ca[t]
    rc = comp.complete_local(b, missing, cb)
    assert all(_bits_equal(x[t], y[t]) for x, y in zip(ra, rc))
    perm = torch.randperm(10, generator=torch.Generator().manual_seed(9))
    perm = perm[perm != t]
    perm = torch.cat([perm[:6], torch.tensor([t]), perm[6:]]).to(DEV)       # the target goes to position 6
    c, cc = a.clone(), ca.clone()
    c[:10], cc[:10] = a[perm], ca[perm]
    rd = comp.complete_local(c, missing, cc)
    assert all(_bits_equal(x[t], y[6]) for x, y in zip(ra, rd))
    assert all(_bits_equal(x[10:], y[10:]) for x, y in zip(ra, rd))


@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_short_catalog_pads_stage_one_and_m0_scores_the_outfit(cat_dtype):
    """A catalog of 3 rows at depth 4: stage 1 pads with -1 and 3^m combinations are scored.  An outfit missing nothing has one
    result, the outfit as given, with its reconstruction error."""
    from codae.tool import OutfitCompleter
    S, E, Q = 3, 64, 6
    model, W, b = _model(S, E, "fp32", 41)
    g = torch.Generator(device=DEV).manual_seed(42)
    cats = _catalogs(S, E, [3, 3, 60], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:4, 0] = True
    missing[2:4, 1] = True
    comp = OutfitCompleter(model, cats, E, depth=4, k=12)
    cand = comp.candidates(outfits, missing)
    assert bool((cand[:4, 0, 3] == -1).all()) and bool((cand[:4, 0, :3] >= 0).all())
    err, ids = comp.complete(outfits, missing, cand)
    nfin = torch.isfinite(err).sum(1).tolist()
    assert nfin == [3, 3, 9, 9, 1, 1], nfin
    ref = _oracle(W, b, model.relu, outfits, missing.cpu(), cand.cpu(), cats, [0] * S, 1.0)
    _check_against_oracle(err, ids, ref, 12, 1e-5)
    assert bool((ids[4:, 0] == -1).all())


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("bad", ["nan", "inf"])
def test_non_finite_input(engine, bad):
    """A NaN in a given slot: every combination's error is NaN, so the outfit gets (+inf, -1) throughout.  A NaN or inf candidate row:
    its combinations are NaN (never ranked) or +inf (after every finite one).  Other outfits are bit-identical to a clean run."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 3, 64, 12, 4
    model, _, _ = _model(S, E, engine, 51)
    g = torch.Generator(device=DEV).manual_seed(52)
    cats = _catalogs(S, E, [40, 40, 40], torch.float32, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 2] = True
    missing[::2, 1] = True
    cand = torch.randint(0, 40, (Q, S, depth), generator=g, device=DEV)
    cand[5, 2, 1] = 7
    comp = OutfitCompleter(model, cats, E, depth=depth, k=16, chunk=100)
    ra = [x.clone() for x in comp.complete_local(outfits, missing, cand)]
    x = outfits.clone()
    x[3, 0 * E + 5] = float("nan")
    err, ids = (t.clone() for t in comp.complete_local(x, missing, cand))
    assert bool(torch.isinf(err[3]).all()) and bool((ids[3] == -1).all())
    keep = torch.arange(Q, device=DEV) != 3
    assert _bits_equal(err[keep], ra[0][keep]) and _bits_equal(ids[keep], ra[1][keep])
    cats2 = [c.clone() for c in cats]
    cats2[2][7, 3] = float(bad)
    comp2 = OutfitCompleter(model, cats2, E, depth=depth, k=16, chunk=100)
    err, ids = comp2.complete_local(outfits, missing, cand)
    hit = (cand[:, 2] == 7).any(1)
    for q in range(Q):
        if not bool(hit[q]):
            assert _bits_equal(err[q], ra[0][q]) and _bits_equal(ids[q], ra[1][q])
            continue
        has7 = ids[q, :, 2] == 7
        fin = torch.isfinite(err[q])
        assert not bool((has7 & fin).any())                          # never ranked among the finite errors
        n_fin = int(fin.sum())
        assert bool(torch.isinf(err[q][has7]).all()) and bool((~fin[:n_fin]).sum() == 0)


def _planted_model(S, E, engine):
    """Square layers (z = io), every Linear the identity but the last, which maps every slot to the mean of all slots: the
    reconstruction error of an outfit is zero exactly when its slots are equal.  Inputs are >= 0, so the ReLUs pass."""
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
def test_planted_completion(engine, cat_dtype):
    """Given slots hold copies of one item v; each missing slot's catalog holds a copy of v among random distractors.  The stage-1
    reading (the mean of the given slots, a multiple of v) finds the copies by cosine, and the best completion is the planted rows
    with error ~ 0."""
    from codae.tool import OutfitCompleter
    S, E, Q, n = 4, 32, 40, 300
    model = _planted_model(S, E, engine)
    g = torch.Generator(device=DEV).manual_seed(61)
    v = torch.rand((Q, E), generator=g, device=DEV).to(torch.bfloat16).float()          # exact in both catalog dtypes
    outfits = v.repeat(1, S)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 1] = True
    missing[::2, 3] = True
    cats, planted = [], []
    for s in range(S):
        cat = torch.rand((n, E), generator=g, device=DEV)
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(s))[:Q].to(DEV)
        cat[rows] = v
        cats.append(cat.to(cat_dtype))
        planted.append(rows)
    comp = OutfitCompleter(model, cats, E, depth=4, k=3, metric="cosine")
    err, ids = comp.complete(outfits, missing, None)
    assert bool((err[:, 0] <= 1e-4).all()), err[:, 0].max()
    for s in (1, 3):
        want = torch.where(missing[:, s], planted[s], -1)
        assert torch.equal(ids[:, 0, s], want), s
    assert bool((ids[:, 0, 0] == -1).all()) and bool((ids[:, 0, 2] == -1).all())
    assert bool((err[:, 1] > 1e-3).all())


def _guarded(bufs, nbytes, guard=4096, fill=255):            # 0xff bytes: NaN as float32 / bf16, -1 as integers
    buf = torch.full((guard + nbytes + guard,), fill, dtype=torch.uint8, device=DEV)
    bufs.append(buf)
    return buf[guard:guard + nbytes]


def test_outputs_stay_in_bounds_and_bad_arguments_are_rejected():
    """Built rows and errors inside NaN-filled guarded allocations: rows b < B, columns < io and err[pos[b]] of valid combinations
    are written, nothing else.  Bad device data (a position outside [0, Q C), c >= depth^m_q, slot_base past the pool, pool_id < 0)
    gives a zero row and no error.  CODAE_EINVAL for bad host arguments."""
    from codae import _C
    S, E, Q, depth, guard = 3, 64, 5, 4, 4096
    io, C = S * E, 16
    g = torch.Generator(device=DEV).manual_seed(71)
    outfits = torch.rand((Q, io), generator=g, device=DEV)
    pool = torch.rand((Q * 2 * depth, E), generator=g, device=DEV)
    pool_id = torch.arange(pool.shape[0], dtype=torch.int64, device=DEV) + 1000
    pool_id[9] = -1
    slot_base = torch.full((Q, S), -1, dtype=torch.int64, device=DEV)
    slot_base[:, 0] = torch.arange(Q, device=DEV) * 2 * depth
    slot_base[:, 2] = torch.arange(Q, device=DEV) * 2 * depth + depth
    slot_base[4, 2] = pool.shape[0] - 2                              # candidate 2.. of outfit 4, slot 2 lie past the pool
    slot_base[3, 0] = -1                                             # outfit 3 misses one slot: c >= 4 is invalid
    pos = torch.tensor([0, 5, 1 * C + 1 * 4 + 1, 1 * C + 2, 3 * C + 3, 3 * C + 4, 4 * C + 4 * 2, 4 * C + 4, -1, Q * C, 2 * C + 15],
                       dtype=torch.int64, device=DEV)
    valid = [True, True, False, True, True, False, False, True, False, False, True]          # pos 1*C+5 takes pool row 9
    B = pos.numel()
    ld_x = io + 64
    for xdt, esz in ((torch.float32, 4), (torch.bfloat16, 2)):
        bufs = []
        x = _guarded(bufs, B * ld_x * esz).view(xdt).view(B, ld_x)
        err = _guarded(bufs, Q * C * 4).view(torch.float32)
        before = [t.clone() for t in bufs]
        _C.complete_build(outfits, S, E, slot_base, pool, pool_id, depth, C, pos, 0.5, x)
        y = torch.rand((B, io), generator=g, device=DEV)
        _C.complete_error(outfits, S, E, slot_base, pool, pool_id, depth, C, pos, 0.5, y, err)
        torch.cuda.synchronize()
        for bb, b0 in zip(bufs, before):
            assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])
        assert bool(torch.isnan(x[:, io:].float()).all())
        wrote = torch.zeros(Q * C, dtype=torch.bool)
        for b_, (p, ok) in enumerate(zip(pos.tolist(), valid)):
            row = x[b_, :io].float()
            if not ok:
                assert not bool(row.any()), b_
                continue
            q, c = divmod(p, C)
            want = outfits[q].clone()
            j = 0
            for s in range(S):
                base = int(slot_base[q, s])
                if base < 0:
                    continue
                want[s * E:(s + 1) * E] = pool[base + (c // depth ** j) % depth] * 0.5
                j += 1
            assert torch.equal(row, want.to(xdt).float()), b_
            xe = want
            wrote[p] = True
            e_ref = ((y[b_] - xe) ** 2).sum()
            assert abs(float(err[p]) - float(e_ref)) <= 1e-5 * float(e_ref), b_
        assert bool(torch.isnan(err.cpu()[~wrote]).all())
    c, L, P, st = _C.ctx(DEV), _C.lib(), _C.p, _C.stream()
    x = torch.empty((B, io), device=DEV)
    err = torch.empty(Q * C, device=DEV)

    def call(fn, **kw):
        a = dict(o=P(outfits), ldo=io, Q=Q, S=S, E=E, sb=P(slot_base), pool=P(pool), ldp=E, R=pool.shape[0], pid=P(pool_id),
                 depth=depth, C=C, pos=P(pos), B=B, x=P(x), xdt=_C.F32, ldx=io, y=P(x), ldy=io, err=P(err))
        a.update(kw)
        head = (c, a["o"], a["ldo"], a["Q"], a["S"], a["E"], a["sb"], a["pool"], a["ldp"], a["R"], a["pid"], a["depth"], a["C"],
                a["pos"], a["B"], 0.5)
        if fn == "build":
            return L.codae_complete_build(*head, a["x"], a["xdt"], a["ldx"], st)
        return L.codae_complete_error(*head, a["y"], a["ldy"], a["err"], st)
    for fn in ("build", "error"):
        assert call(fn) == _C.OK
        common = (dict(o=None), dict(sb=None), dict(pool=None), dict(pid=None), dict(pos=None), dict(Q=0), dict(S=0), dict(S=65),
                  dict(E=0), dict(B=0), dict(depth=0), dict(depth=129), dict(C=0), dict(C=4097), dict(Q=2 ** 20, C=4096),
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
    model, _, _ = _model(S, E, "bf16", 81)
    cats = [torch.rand((20, E), device=DEV), None, torch.rand((20, E), device=DEV)]
    for kw in (dict(depth=0), dict(depth=129), dict(k=0), dict(k=129)):
        with pytest.raises(RuntimeError):
            OutfitCompleter(model, cats, E, **kw)
    comp = OutfitCompleter(model, cats, E, depth=17)
    o = torch.rand((4, S * E), device=DEV)
    m = torch.zeros((4, S), dtype=torch.bool, device=DEV)
    m[0, [0, 2]] = True
    with pytest.raises(RuntimeError, match="no catalog"):
        comp.complete(o, m | torch.tensor([False, True, False], device=DEV))
    with pytest.raises(RuntimeError, match="combinations"):
        comp.complete_local(o, m, torch.zeros((4, S, 65), dtype=torch.int64, device=DEV))
    for bad, match in (((o.double(), m), "float32"), ((o.cpu(), m), "device"), ((o, m.cpu()), "device"), ((o, m.int()), "bool"),
                       ((o, m[:, :2]), "shape")):
        with pytest.raises(RuntimeError, match=match):
            comp.complete(*bad)
    with pytest.raises(RuntimeError, match="device"):
        comp.complete_local(o, m, torch.zeros((4, S, 4), dtype=torch.int64))


@pytest.mark.parametrize("engine", ["bf16", "fp32"])
def test_embedding_size(engine):
    """embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)): Q = 256 outfits missing two slots, depth 8 (64 combinations
    each) from 20 000-row bf16 catalogs; 6 outfits checked against fp64."""
    from codae.tool import OutfitCompleter
    S, E, Q = 3, 512, 256
    model, W, b = _model(S, E, engine, 91, z=1536, nin=4, nout=4)
    assert len(model.dims) == 10
    g = torch.Generator(device=DEV).manual_seed(92)
    cats = _catalogs(S, E, [20_000] * 3, torch.bfloat16, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 1:] = True
    comp = OutfitCompleter(model, cats, E, depth=8, k=10)
    cand = comp.candidates(outfits, missing)
    err, ids = comp.complete(outfits, missing, cand)
    assert bool(torch.isfinite(err).all()) and bool((ids[:, :, 1:] >= 0).all())
    pick = [0, 17, 63, 128, 200, 255]
    ref = _oracle(W, b, model.relu, outfits[pick], missing[pick].cpu(), cand[pick].cpu(), cats, [0] * S, 1.0)
    _check_against_oracle(err[pick], ids[pick], ref, 10, RTOL[engine])


def test_script_complete_mode(tmp_path):
    args = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config", os.path.join(PKG, "config", "embedding.yaml"),
            "--synthetic", "3000", "--queries", "16", "--mode", "complete", "--missing", "1,2", "--complete_depth", "4",
            "--k", "5", "--dtype", "bf16", "--catalog_dtype", "bf16"]
    r = subprocess.run([sys.executable] + args, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["mode"] == "complete" and res["missing"] == [1, 2] and res["depth"] == 4
    assert len(res["ids"]) == 16 and all(len(x) == 5 and all(len(t) == 3 for t in x) for x in res["ids"])
    assert all(t[0] == -1 and t[1] >= 0 and t[2] >= 0 for x in res["ids"] for t in x)
    assert all(row == sorted(row) for row in res["errors"])
    for flag in (["--exclude_own_item"], ["--allowed_rows", "x.npy"]):
        r = subprocess.run([sys.executable] + args + flag, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
        assert r.returncode != 0 and "complete" in r.stderr


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
missing = (torch.rand((Q, S), generator=gen) < 0.5).to(dev)
missing[:, 0] = True
lo, n = shard_rows(N, G, r)
comp = OutfitCompleter(model, [c[lo:lo + n] for c in full], E, depth=4, k=6, row_offsets=[lo] * S, chunk=300)
one = OutfitCompleter(model, full, E, depth=4, k=6, chunk=300, process_group=None)
cand = comp.candidates(outfits, missing)
err, ids = (t.clone() for t in comp.complete(outfits, missing, cand))
assert err.shape == (Q, 6) and ids.shape == (Q, 6, S)
for q in range(G):
    a, m = shard_rows(Q, G, q)
    e, i = one.complete_local(outfits[a:a + m], missing[a:a + m], cand[a:a + m])
    assert torch.equal(e.view(torch.int32), err[a:a + m].view(torch.int32)) and torch.equal(i, ids[a:a + m]), q
# stage-1 ids equal the single-GPU ids: the full-catalog completer runs its stage 1 once the process group is gone
dist.barrier()
dist.destroy_process_group()
c1 = one.candidates(outfits, missing)
assert torch.equal(c1, cand)
if r == 0:
    print("COMPLETE DIST OK")
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_complete_on_two_gpus(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "complete_dist.py"
    script.write_text(DIST)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), PKG]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "COMPLETE DIST OK" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
