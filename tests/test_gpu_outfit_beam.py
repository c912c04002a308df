"""GPU tests of outfit completion by beam search (codae_complete_beam_build / codae_complete_beam_error; OutfitCompleter.complete_beam_local
/ complete_beam; 4_complementarity_inference.py --mode complete --beam).  The missing slots are filled one level at a time and the
best W partial outfits are kept after each; a GEMM row depends only on that row and on the launch's 128-row tile count, so at chunks
of <= 128 rows a beam that holds every combination is exhaustive completion bit for bit."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import PKG
from test_gpu_outfit_complete import _bits_equal, _catalogs, _guarded, _model

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ENGINES = ["fp32", "fp32_simt", "bf16"]
RTOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-2}
CAT_DTYPES = [torch.float32, torch.bfloat16]


def _mixed_missing(Q, S, seed):
    missing = torch.zeros((Q, S), dtype=torch.bool)
    for q in range(Q):
        missing[q, torch.randperm(S, generator=torch.Generator().manual_seed(seed + q))[:q % 4]] = True
    return missing.to(DEV)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_no_pruning_is_exhaustive_bit_for_bit(engine, cat_dtype):
    """W >= depth^(m_max - 1) and chunk <= 128: complete_beam_local is complete_local, errors and ids, with m_q = 0..3 in one call,
    padding ids, ids outside the catalogs and an outfit whose missing slot has no valid candidate."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 4, 32, 24, 4
    model, _, _ = _model(S, E, engine, 101)
    g = torch.Generator(device=DEV).manual_seed(102)
    cats = _catalogs(S, E, [30 + 7 * s for s in range(S)], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = _mixed_missing(Q, S, 0)
    cand = torch.randint(-1, 45, (Q, S, depth), generator=g, device=DEV)
    cand[7] = -1                                                  # outfit 7 (m_q = 3): every expansion invalid
    for chunk, W, k in ((128, 16, 10), (37, 16, 16), (128, 64, 5)):
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, inv_scale=0.5, chunk=chunk)
        e1, i1 = (t.clone() for t in comp.complete_local(outfits, missing, cand))
        e2, i2 = comp.complete_beam_local(outfits, missing, cand, W)
        assert _bits_equal(e1, e2) and _bits_equal(i1, i2), (chunk, W)
        assert bool(torch.isinf(e2[7]).all()) and bool((i2[7] == -1).all())
        e3, i3 = comp.complete_beam(outfits, missing, W, cand)
        assert _bits_equal(e2, e3) and _bits_equal(i2, i3)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("cat_dtype", CAT_DTYPES)
def test_one_missing_slot_is_complete_and_rerank(engine, cat_dtype):
    from codae.tool import OutfitCompleter, SwapScorer
    S, E, Q, depth, k = 3, 64, 300, 8, 5
    model, _, _ = _model(S, E, engine, 111)
    g = torch.Generator(device=DEV).manual_seed(112)
    cats = _catalogs(S, E, [400, 400, 400], cat_dtype, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 1] = True
    comp = OutfitCompleter(model, cats, E, depth=depth, k=k, inv_scale=0.7, chunk=1000)
    cand = comp.candidates(outfits, missing)
    e1, i1 = (t.clone() for t in comp.complete(outfits, missing, cand))
    e2, i2 = comp.complete_beam(outfits, missing, 6, cand)
    assert _bits_equal(e1, e2) and _bits_equal(i1, i2)
    ws, wi = SwapScorer(model, cats[1], E, k=k, inv_scale=0.7, chunk=1000).rerank(outfits, 1, cand[:, 1].contiguous())
    assert _bits_equal(e2, ws) and torch.equal(i2[:, :, 1], wi)


def _beam_ref(outfits, slot_base, pool, pool_id, beam_c, depth, level, p, inv_scale):
    """Restatement of one child: (valid, x' [io] fp32 with hidden slots 0, visible column mask [io])."""
    Q, S = slot_base.shape
    io = outfits.shape[1]
    E = io // S
    W = beam_c.shape[1]
    x = torch.zeros(io, device=DEV)
    vis = torch.zeros(io, dtype=torch.bool, device=DEV)
    if p < 0 or p >= Q * W * depth:
        return False, x, vis
    q, t, b = p // (W * depth), (p // depth) % W, p % depth
    parent = int(beam_c[q, t])
    if parent < 0:
        return False, x, vis
    ms = [s for s in range(S) if int(slot_base[q, s]) >= 0]
    if level >= len(ms) or parent >= depth ** level:
        return False, x, vis
    c = parent + b * depth ** level
    x = outfits[q].clone()
    vis[:] = True
    for j, s in enumerate(ms):
        if j > level:
            x[s * E:(s + 1) * E] = 0.0
            vis[s * E:(s + 1) * E] = False
            continue
        r = int(slot_base[q, s]) + (c // depth ** j) % depth
        if r >= pool.shape[0] or int(pool_id[r]) < 0:
            return False, torch.zeros(io, device=DEV), torch.zeros(io, dtype=torch.bool, device=DEV)
        x[s * E:(s + 1) * E] = pool[r] * inv_scale
    return True, x, vis


def test_kernel_contract_at_every_level():
    """The two C entry points driven directly for random parents (some empty, some >= depth^level) at every level: built rows exact
    (hidden slots +0.0, padding, short pools, unowned rows and bad parents or levels are zero rows), err against an fp64 restatement
    of the partial error, rows not built stay NaN, nothing written outside the outputs (guarded allocations); CODAE_EINVAL for bad
    host arguments."""
    from codae import _C
    S, E, Q, depth, W, guard = 4, 32, 6, 3, 4, 4096
    io = S * E
    g = torch.Generator(device=DEV).manual_seed(121)
    outfits = torch.rand((Q, io), generator=g, device=DEV)
    npool = Q * S * depth
    pool = torch.rand((npool, E), generator=g, device=DEV)
    pool_id = torch.arange(npool, dtype=torch.int64, device=DEV) + 500
    pool_id[torch.randperm(npool, generator=torch.Generator().manual_seed(1))[:8].to(DEV)] = -1
    missing = _mixed_missing(Q, S, 40) | (torch.arange(Q, device=DEV) == 3).view(-1, 1)      # outfit 3 misses all four
    slot_base = torch.where(missing, torch.arange(Q * S, device=DEV).view(Q, S) * depth, -1)
    slot_base[5, 3] = npool - 1 if bool(missing[5, 3]) else -1                             # candidates 1, 2 past the pool
    G = Q * W * depth
    pos = torch.cat([torch.arange(G, dtype=torch.int64, device=DEV), torch.tensor([-1, G, G + 5], device=DEV)])
    pos = pos[torch.randperm(pos.numel(), generator=torch.Generator().manual_seed(2)).to(DEV)]
    B = pos.numel()
    ld_x = io + 64
    for level in range(S):
        beam_c = torch.randint(-1, depth ** level + 2, (Q, W), generator=g, device=DEV)
        y = torch.rand((B, io), generator=g, device=DEV)
        for xdt, esz in ((torch.float32, 4), (torch.bfloat16, 2)):
            bufs = []
            x = _guarded(bufs, B * ld_x * esz).view(xdt).view(B, ld_x)
            err = _guarded(bufs, G * 4).view(torch.float32)
            before = [t.clone() for t in bufs]
            _C.complete_beam_build(outfits, S, E, slot_base, pool, pool_id, depth, beam_c, level, pos, 0.5, x)
            _C.complete_beam_error(outfits, S, E, slot_base, pool, pool_id, depth, beam_c, level, pos, 0.5, y, err)
            torch.cuda.synchronize()
            for bb, b0 in zip(bufs, before):
                assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])
            assert bool(torch.isnan(x[:, io:].float()).all())
            wrote = torch.zeros(G, dtype=torch.bool)
            n_valid = 0
            for b_, p in enumerate(pos.tolist()):
                ok, want, vis = _beam_ref(outfits, slot_base, pool, pool_id, beam_c, depth, level, p, 0.5)
                row = x[b_, :io].float()
                assert _bits_equal(row, want.to(xdt).float()), (level, b_, p, ok)
                if not ok:
                    continue
                n_valid += 1
                wrote[p] = True
                e_ref = float((((y[b_].double() - want.double()) ** 2) * vis.double()).sum())
                assert abs(float(err[p]) - e_ref) <= 1e-5 * e_ref, (level, b_)
            assert bool(torch.isnan(err.cpu()[~wrote]).all())
            assert n_valid > 0 or level == S - 1, level
    c, L, P, st = _C.ctx(DEV), _C.lib(), _C.p, _C.stream()
    beam_c = torch.zeros((Q, W), dtype=torch.int64, device=DEV)
    x = torch.empty((B, io), device=DEV)
    err = torch.empty(G, device=DEV)

    def call(fn, **kw):
        a = dict(o=P(outfits), ldo=io, Q=Q, S=S, E=E, sb=P(slot_base), pool=P(pool), ldp=E, R=npool, pid=P(pool_id), depth=depth,
                 bc=P(beam_c), W=W, level=1, pos=P(pos), B=B, x=P(x), xdt=_C.F32, ldx=io, y=P(x), ldy=io, err=P(err))
        a.update(kw)
        head = (c, a["o"], a["ldo"], a["Q"], a["S"], a["E"], a["sb"], a["pool"], a["ldp"], a["R"], a["pid"], a["depth"], a["bc"],
                a["W"], a["level"], a["pos"], a["B"], 0.5)
        if fn == "build":
            return L.codae_complete_beam_build(*head, a["x"], a["xdt"], a["ldx"], st)
        return L.codae_complete_beam_error(*head, a["y"], a["ldy"], a["err"], st)
    for fn in ("build", "error"):
        assert call(fn) == _C.OK
        common = (dict(o=None), dict(sb=None), dict(pool=None), dict(pid=None), dict(bc=None), dict(pos=None), dict(Q=0), dict(S=0),
                  dict(S=65), dict(E=0), dict(B=0), dict(depth=0), dict(depth=129), dict(W=0), dict(W=129), dict(level=-1),
                  dict(level=S), dict(S=12, E=1, depth=128, level=8), dict(Q=2 ** 20, W=128, depth=16), dict(R=0), dict(ldp=E - 1),
                  dict(ldo=io - 1), dict(o=outfits.data_ptr() + 2), dict(sb=slot_base.data_ptr() + 4), dict(bc=beam_c.data_ptr() + 4),
                  dict(pid=pool_id.data_ptr() + 4), dict(pos=pos.data_ptr() + 4), dict(pool=pool.data_ptr() + 2))
        extra = ((dict(x=None), dict(ldx=io - 1), dict(xdt=7), dict(x=x.data_ptr() + 1)) if fn == "build" else
                 (dict(y=None), dict(err=None), dict(ldy=io - 1), dict(err=err.data_ptr() + 2)))
        for kw in common + extra:
            assert call(fn, **kw) == _C.EINVAL, (fn, kw)
    torch.cuda.synchronize()


def _dae64(W, b, relu, x):
    """fp64 forward of the model's weights (W, b as _model returns them) on rows x [n, io]."""
    h = x.double()
    for w, v, rl in zip(W, b, relu):
        h = h @ w.to(DEV).double().T + v.to(DEV).double()
        if rl:
            h = torch.relu(h)
    return h


@pytest.mark.parametrize("engine", ENGINES)
def test_width_one_is_greedy(engine):
    """W = 1 against an explicit greedy restatement in fp64: at each level the beam's pick has the smallest partial error among the
    candidates of that slot (up to the engine's tolerance), given the earlier picks and the later slots hidden as zeros; the returned
    error is the fp64 error of the completed outfit."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 5, 32, 12, 6
    model, Wt, bt = _model(S, E, engine, 131)
    g = torch.Generator(device=DEV).manual_seed(132)
    cats = _catalogs(S, E, [60] * S, torch.float32, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, [0, 2, 4]] = True
    missing[::3, 1] = True
    cand = torch.stack([torch.randperm(60, generator=torch.Generator().manual_seed(q))[:S * depth].view(S, depth)
                        for q in range(Q)]).to(DEV)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=1, chunk=128)
    err, ids = comp.complete_beam_local(outfits, missing, cand, 1)
    tol = 4 * RTOL[engine]
    for q in range(Q):
        ms = [s for s in range(S) if missing[q, s]]
        x = outfits[q].clone()
        for s in ms:
            x[s * E:(s + 1) * E] = 0.0
        for j, s in enumerate(ms):
            rows = x.repeat(depth, 1)
            for b in range(depth):
                rows[b, s * E:(s + 1) * E] = cats[s][int(cand[q, s, b])]
            vis = torch.ones(S * E, dtype=torch.bool, device=DEV)
            for s2 in ms[j + 1:]:
                vis[s2 * E:(s2 + 1) * E] = False
            pe = (((_dae64(Wt, bt, model.relu, rows) - rows.double()) ** 2) * vis.double()).sum(1)
            pick = int(ids[q, 0, s])
            b_pick = int((cand[q, s] == pick).nonzero()[0])
            assert float(pe[b_pick]) <= float(pe.min()) * (1 + tol) + 1e-6, (q, j, pe.tolist(), b_pick)
            x[s * E:(s + 1) * E] = cats[s][pick]
        full = float(((_dae64(Wt, bt, model.relu, x.view(1, -1)) - x.double()) ** 2).sum())
        assert abs(float(err[q, 0]) - full) <= RTOL[engine] * full, (q, float(err[q, 0]), full)


@pytest.mark.parametrize("engine", ENGINES)
def test_independent_of_other_outfits_and_repeatable(engine):
    from codae.tool import OutfitCompleter
    S, E, Q, depth, t = 4, 32, 20, 5, 6
    model, _, _ = _model(S, E, engine, 141)
    g = torch.Generator(device=DEV).manual_seed(142)
    cats = _catalogs(S, E, [50] * S, torch.float32, g)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=4, chunk=128)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 1:] = True
    a = torch.rand((Q, S * E), generator=g, device=DEV)
    ca = torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    ra = [x.clone() for x in comp.complete_beam_local(a, missing, ca, 4)]
    rb = comp.complete_beam_local(a, missing, ca, 4)
    assert all(_bits_equal(x, y) for x, y in zip(ra, rb))
    b, cb = torch.rand((Q, S * E), generator=g, device=DEV), torch.randint(0, 50, (Q, S, depth), generator=g, device=DEV)
    b[t], cb[t] = a[t], ca[t]
    mb = missing.clone()
    mb[::2, 2] = False                                            # other outfits end at other levels
    mb[t] = True
    mb[t, 0] = False
    rc = comp.complete_beam_local(b, mb, cb, 4)
    assert all(_bits_equal(x[t], y[t]) for x, y in zip(ra, rc))
    rd = comp.complete_beam_local(a[t:t + 1], missing[t:t + 1], ca[t:t + 1], 4)
    assert all(_bits_equal(x[t], y[0]) for x, y in zip(ra, rd))


@pytest.mark.parametrize("engine", ENGINES)
def test_polyvore_shape_seven_of_eight(engine):
    """8 slots, 7 missing, depth 16 (16^7 combinations, far past complete's cap), W = 16: each returned combination fed back to
    complete_local as a depth-1 candidate list gives the same error bit for bit; errors are sorted, ties -> lower c.  Every launch of
    the beam has 128 rows (Q W depth = 2048 per level, 128 at level 0), and the fed-back combinations go in one launch of 128 rows too:
    the FFMA engine's plan follows the row count (split-K from M N >= 64 x 64 when K >= 256).  Stage 1 runs without the exhaustive
    cap when complete_beam is given no candidates."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth, W, k = 8, 32, 8, 16, 16, 8
    model, _, _ = _model(S, E, engine, 151, z=128)
    g = torch.Generator(device=DEV).manual_seed(152)
    cats = _catalogs(S, E, [200] * S, torch.bfloat16, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.ones((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 0] = False
    cand = torch.stack([torch.randperm(200, generator=torch.Generator().manual_seed(q))[:S * depth].view(S, depth)
                        for q in range(Q)]).to(DEV)
    comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=128)
    with pytest.raises(RuntimeError, match="combinations"):
        comp.complete_local(outfits, missing, cand)
    err, ids = (t.clone() for t in comp.complete_beam_local(outfits, missing, cand, W))
    assert bool(torch.isfinite(err).all()) and bool((ids[:, :, 1:] >= 0).all()) and bool((ids[:, :, 0] == -1).all())
    one = OutfitCompleter(model, cats, E, depth=1, k=1, chunk=128)
    rep = 128 // (Q * k)
    fed = ids.reshape(Q * k, S, 1).repeat(rep, 1, 1)                                         # rows (q, e), twice
    e1, i1 = one.complete_local(outfits.repeat_interleave(k, 0).repeat(rep, 1), missing[:1].expand(128, S).contiguous(), fed)
    assert _bits_equal(e1[:, 0], err.reshape(-1).repeat(rep)) and torch.equal(i1[:, 0], ids.reshape(Q * k, S).repeat(rep, 1))
    e2, i2 = comp.complete_beam(outfits, missing, W)                                        # stage 1 included
    assert e2.shape == (Q, k) and bool(torch.isfinite(e2).all()) and bool((i2[:, :, 1:] >= 0).all())
    digit = (cand.unsqueeze(1) == ids.unsqueeze(3)).to(torch.int64).argmax(3)             # [Q, k, S]
    c = (digit[:, :, 1:] * depth ** torch.arange(S - 1, device=DEV)).sum(2)
    for q in range(Q):
        for e in range(k - 1):
            assert float(err[q, e]) < float(err[q, e + 1]) or (err[q, e] == err[q, e + 1] and c[q, e] < c[q, e + 1]), (q, e)


@pytest.mark.parametrize("engine", ENGINES)
def test_non_finite_input(engine):
    """NaN in a given slot: (+inf, -1) throughout.  inf in a given slot: every returned error is +inf.  A NaN candidate row is never
    returned, and with no pruning the beam still equals complete_local bit for bit."""
    from codae.tool import OutfitCompleter
    S, E, Q, depth = 3, 64, 12, 4
    model, _, _ = _model(S, E, engine, 161)
    g = torch.Generator(device=DEV).manual_seed(162)
    cats = _catalogs(S, E, [40, 40, 40], torch.float32, g)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    missing = torch.zeros((Q, S), dtype=torch.bool, device=DEV)
    missing[:, 2] = True
    missing[::2, 1] = True
    cand = torch.randint(0, 40, (Q, S, depth), generator=g, device=DEV)
    cand[5, 2, 1] = 7
    comp = OutfitCompleter(model, cats, E, depth=depth, k=4, chunk=100)
    ra = [t.clone() for t in comp.complete_beam_local(outfits, missing, cand, 4)]
    for bad in ("nan", "inf"):
        x = outfits.clone()
        x[3, 0 * E + 5] = float(bad)
        err, ids = comp.complete_beam_local(x, missing, cand, 4)
        if bad == "nan":
            assert bool(torch.isinf(err[3]).all()) and bool((ids[3] == -1).all())
        else:
            assert bool((err[3] == float("inf")).all())
        keep = torch.arange(Q, device=DEV) != 3
        assert _bits_equal(err[keep], ra[0][keep]) and _bits_equal(ids[keep], ra[1][keep])
    cats2 = [c.clone() for c in cats]
    cats2[2][7, 3] = float("nan")
    comp2 = OutfitCompleter(model, cats2, E, depth=depth, k=4, chunk=100)
    e1, i1 = (t.clone() for t in comp2.complete_local(outfits, missing, cand))
    e2, i2 = comp2.complete_beam_local(outfits, missing, cand, 4)
    assert _bits_equal(e1, e2) and _bits_equal(i1, i2)
    assert not bool((i2[:, :, 2] == 7).any())


def test_limits_raise_before_any_launch():
    from codae.tool import OutfitCompleter
    S, E = 3, 64
    model, _, _ = _model(S, E, "bf16", 171)
    cats = [torch.rand((20, E), device=DEV), None, torch.rand((20, E), device=DEV)]
    comp = OutfitCompleter(model, cats, E, depth=4, k=4)
    o = torch.rand((4, S * E), device=DEV)
    m = torch.zeros((4, S), dtype=torch.bool, device=DEV)
    m[0, [0, 2]] = True
    cand = torch.zeros((4, S, 4), dtype=torch.int64, device=DEV)
    for w, match in ((0, "width"), (129, "width"), (3, "exceeds the beam width")):
        with pytest.raises(RuntimeError, match=match):
            comp.complete_beam(o, m, w)
        with pytest.raises(RuntimeError, match=match):
            comp.complete_beam_local(o, m, cand, w)
    with pytest.raises(RuntimeError, match="no catalog"):
        comp.complete_beam(o, m | torch.tensor([False, True, False], device=DEV), 4)
    with pytest.raises(RuntimeError, match="device"):
        comp.complete_beam_local(o, m, cand.cpu(), 4)


def test_script_complete_beam_mode(tmp_path):
    base = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config", os.path.join(PKG, "config", "embedding.yaml"),
            "--synthetic", "3000", "--queries", "16", "--mode", "complete", "--missing", "1,2", "--complete_depth", "4",
            "--k", "5", "--dtype", "bf16", "--catalog_dtype", "bf16"]
    out = {}
    for extra in ([], ["--beam", "16"], ["--beam", "5"]):
        r = subprocess.run([sys.executable] + base + extra, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        out[len(extra) and int(extra[1])] = json.loads(r.stdout.strip().splitlines()[-1])
    assert "beam" not in out[0] and out[16]["beam"] == 16 and out[5]["beam"] == 5
    res = out[5]
    assert len(res["ids"]) == 16 and all(len(x) == 5 and all(len(t) == 3 for t in x) for x in res["ids"])
    assert all(t[0] == -1 and t[1] >= 0 and t[2] >= 0 for x in res["ids"] for t in x)
    assert all(row == sorted(row) for row in res["errors"])


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
S, E, Q, N = 4, 64, 101, 500
torch.manual_seed(5)
model = EmbeddingDenoisingAutoencoder(S * E, 96, E, 2, 2, False).to(dev).set_compute_dtype("bf16")
gen = torch.Generator().manual_seed(6)
outfits = torch.rand((Q, S * E), generator=gen).to(dev)
full = [torch.rand((N, E), generator=gen).to(dev) for _ in range(S)]
missing = (torch.rand((Q, S), generator=gen) < 0.6).to(dev)
missing[0] = False
lo, n = shard_rows(N, G, r)
comp = OutfitCompleter(model, [c[lo:lo + n] for c in full], E, depth=6, k=4, row_offsets=[lo] * S, chunk=128)
one = OutfitCompleter(model, full, E, depth=6, k=4, chunk=128, process_group=None)
cand = comp.candidates(outfits, missing)
err, ids = (t.clone() for t in comp.complete_beam(outfits, missing, 8, cand))
assert err.shape == (Q, 4) and ids.shape == (Q, 4, S)
e1, i1 = one.complete_beam_local(outfits, missing, cand, 8)
assert torch.equal(e1.view(torch.int32), err.view(torch.int32)) and torch.equal(i1, ids)
dist.barrier()
dist.destroy_process_group()
if r == 0:
    print("BEAM DIST OK")
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_complete_beam_on_two_gpus(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "beam_dist.py"
    script.write_text(DIST)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), PKG]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "BEAM DIST OK" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
