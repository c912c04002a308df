"""GPU tests of swap scoring over per-outfit candidate lists (codae_swap_build_pairs, codae_swap_error_pairs,
codae_swap_pairs_topk; SwapScorer.rerank_local / rerank).  A pair's error is computed as SwapScorer.topk_local computes a
candidate's, and the tensor-core GEMM plan depends on a launch's row count M only through its 128-row tile count ceil(M / 128)
(make_plan / pick_bn in csrc/gemm_tcgen05.cu): chunks with the same tile counts give the same bits, other layouts agree to the
engine's tolerance."""
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
ENGINES = ["fp32", "fp32_simt", "bf16"]
RTOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-2}
GRID = [(e, b) for e in ENGINES for b in (False, True)]


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
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _oracle_pairs(W, b, relu, outfits, slot, E, cat, cand, inv_scale):
    """fp64-accumulated swap error of every listed pair ([Q, m], NaN for padding / ids outside the catalog)."""
    from oracle import codae_oracle as O
    n = cat.shape[0]
    cand = cand.cpu()
    out = torch.full(cand.shape, float("nan"), dtype=torch.float64)
    for q in range(cand.shape[0]):
        ok = (cand[q] >= 0) & (cand[q] < n)
        if ok.any():
            out[q, ok] = O.score_swaps(W, b, relu, outfits[q], slot, E, cat[cand[q, ok]].float(), inv_scale=inv_scale).cpu()
    return out


def _check_against_oracle(s, i, ref, cand, k, rtol):
    """Returned errors match the oracle pair by pair; the ids are the oracle's top k apart from pairs within tolerance of the k-th
    error (ties by id, NaN never ranks, unused slots (+inf, -1))."""
    s, i = s.cpu(), i.cpu()
    for q in range(cand.shape[0]):
        e = ref[q].numpy()
        ids = cand[q].numpy()
        ok = ~np.isnan(e)
        order = np.lexsort((ids[ok], e[ok]))[:k]
        want_e, want_i = e[ok][order], ids[ok][order]
        n_want = len(want_i)
        assert int((i[q] >= 0).sum()) == n_want, (q, i[q], want_i)
        assert bool(torch.isinf(s[q, n_want:]).all()) and bool((i[q, n_want:] == -1).all())
        got_i = i[q, :n_want].numpy()
        got_s = s[q, :n_want].numpy().astype(np.float64)
        # every returned error is the oracle's error of a listed pair with that id
        for g_s, g_i in zip(got_s, got_i):
            cands = e[ok][ids[ok] == g_i]
            assert len(cands) and np.any(np.abs(cands - g_s) <= rtol * np.abs(cands) + 1e-6), (q, g_i, g_s, cands)
        if n_want:
            kth = want_e[-1]
            tol = rtol * abs(kth) + 1e-6
            for wi, we in zip(want_i, want_e):
                if we < kth - tol:
                    assert wi in got_i, (q, wi, we, kth)
            assert np.all(np.diff(got_s) >= -2 * rtol * np.abs(got_s[1:]) - 1e-6)


@pytest.mark.parametrize("engine,cat_bf16", GRID)
@pytest.mark.parametrize("chunk", [250, 256])
@pytest.mark.parametrize("masked", [False, True])
def test_full_shard_list_equals_topk_local(engine, cat_bf16, chunk, masked):
    """One outfit listing every row of the shard in order: the same errors bit for bit and the same ids as topk_local.  With a
    mask the pair chunks hold the allowed rows only; 60 of 1000 rows are dropped, which leaves every chunk's 128-row tile count as
    in topk_local's row chunks (256 | 256 | 256 | 232 against 256 | 256 | 256 | 172, 4 x 250 against 250 | 250 | 250 | 190)."""
    from codae.tool.inference import SwapScorer
    n, S, E, slot, k, off = 1000, 3, 64, 1, 10, 100
    model, _, _ = _model(S, E, engine, 7)
    torch.manual_seed(8)
    cat = torch.rand(n, E) * 2
    outfit = torch.rand(S * E)
    cat[500:505] = outfit[slot * E:(slot + 1) * E] * 2
    cat[700] = cat[3]                                   # duplicate row: tie -> lower id
    if cat_bf16:
        cat = cat.to(torch.bfloat16)
    allow = None
    if masked:
        allow = torch.ones(n, dtype=torch.bool)
        allow[torch.randperm(n)[:60]] = False
        allow[502] = False
    sc = SwapScorer(model, cat.to(DEV), E, k=k, inv_scale=0.5, row_offset=off, chunk=chunk,
                    allowed=None if allow is None else allow.to(DEV))
    s_ref, i_ref = sc.topk_local(outfit.to(DEV), slot)
    s_ref, i_ref = s_ref.clone(), i_ref.clone()
    cand = torch.arange(off, off + n, dtype=torch.int64, device=DEV).view(1, n)
    s, i = sc.rerank_local(outfit.to(DEV).view(1, -1), slot, cand)
    assert torch.equal(i[0].cpu(), i_ref.cpu()) and _bits_equal(s[0], s_ref)
    if masked:
        assert off + 502 not in i.cpu().tolist()[0]


@pytest.mark.parametrize("engine", ENGINES)
def test_error_does_not_depend_on_other_pairs(engine):
    """Same chunk layout (every entry owned, 5 x 60 pairs, chunk 64); the pairs around pair (2, 10) -- their outfits and ids --
    change, its error stays bit-identical."""
    from codae.tool.inference import SwapScorer
    n, S, E, slot, Q, m = 600, 3, 64, 0, 5, 60
    model, _, _ = _model(S, E, engine, 11)
    torch.manual_seed(12)
    cat = (torch.rand(n, E) * 2).to(DEV)
    sc = SwapScorer(model, cat, E, k=m, chunk=64)
    outfits = torch.rand(Q, S * E, device=DEV)
    cand = torch.randint(0, 300, (Q, m), dtype=torch.int64, device=DEV)
    target = 450
    cand[2, 10] = target
    s_a, i_a = (t.clone() for t in sc.rerank_local(outfits, slot, cand))
    outfits_b = torch.rand(Q, S * E, device=DEV)
    outfits_b[2] = outfits[2]
    cand_b = torch.randint(300, 450, (Q, m), dtype=torch.int64, device=DEV)
    cand_b[2, 10] = target
    s_b, i_b = sc.rerank_local(outfits_b, slot, cand_b)
    ea = s_a[2][i_a[2] == target]
    eb = s_b[2][i_b[2] == target]
    assert ea.numel() == 1 and eb.numel() == 1 and _bits_equal(ea, eb)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("Q,m", [(1, 1), (1, 100), (7, 4), (7, 100), (300, 1), (300, 4), (300, 100)])
@pytest.mark.parametrize("krel", ["below", "equal", "above"])
def test_rerank_matches_oracle(engine, Q, m, krel):
    from codae.tool.inference import SwapScorer
    n, S, E, slot, off = 2000, 3, 64, 2, 0
    k = {"below": max(1, m // 2), "equal": m, "above": min(128, m + 5)}[krel]
    model, W, b = _model(S, E, engine, 21)
    g = torch.Generator().manual_seed(Q * 1000 + m)
    cat = torch.rand(n, E, generator=g) * 2
    outfits = torch.rand(Q, S * E, generator=g)
    cand = torch.randint(0, n, (Q, m), generator=g, dtype=torch.int64)
    cand[torch.rand(Q, m, generator=g) < 0.1] = -1                              # padding
    cand[torch.rand(Q, m, generator=g) < 0.05] = n + 7                          # not in the catalog
    sc = SwapScorer(model, cat.to(DEV), E, k=k, inv_scale=0.5, row_offset=off, chunk=1024)
    s, i = sc.rerank_local(outfits.to(DEV), slot, cand.to(DEV))
    ref = _oracle_pairs(W, b, model.relu, outfits, slot, E, cat, cand, 0.5)
    _check_against_oracle(s, i, ref, cand, k, RTOL[engine])


@pytest.mark.parametrize("cat_bf16", [False, True])
def test_edge_cases(cat_bf16):
    """Padding, all-padding lists, ids outside the catalog and disallowed rows never come back; NaN / inf catalog rows follow the
    sweep's rule (the full list equals topk_local); duplicated ids come back once per listing, consecutively (ties by id)."""
    from codae.tool.inference import SwapScorer
    n, S, E, slot, k = 500, 2, 64, 1, 8
    model, _, _ = _model(S, E, "fp32", 31)
    torch.manual_seed(32)
    cat = torch.rand(n, E) * 2
    cat[40, 3] = float("nan")
    cat[41, 0] = float("inf")
    if cat_bf16:
        cat = cat.to(torch.bfloat16)
    allow = torch.rand(n) < 0.8
    allow[40:42] = True
    allow[7] = False
    sc = SwapScorer(model, cat.to(DEV), E, k=k, chunk=128, allowed=allow.to(DEV))
    outfits = torch.rand(4, S * E, device=DEV)
    full = torch.arange(n, dtype=torch.int64, device=DEV).view(1, n)
    s, i = sc.rerank_local(outfits[:1], slot, full)
    s_ref, i_ref = sc.topk_local(outfits[0], slot)
    assert torch.equal(i[0], i_ref) and _bits_equal(s[0], s_ref)
    assert 40 not in i.tolist()[0]
    ok_row = int(torch.nonzero(allow[100:]).flatten()[0]) + 100
    cand = torch.tensor([[-1] * 6,                                      # all padding
                         [7, -3, n, n + 100, 40, -1],                   # disallowed, padding, outside, NaN row
                         [ok_row, ok_row, 7, ok_row, 5000, -1],         # duplicates
                         [41, ok_row, -1, -1, -1, -1]], dtype=torch.int64, device=DEV)
    s, i = (t.cpu() for t in sc.rerank_local(outfits, slot, cand))
    assert i[0].tolist() == [-1] * k and bool(torch.isinf(s[0]).all())
    assert i[1].tolist() == [-1] * k
    assert i[2].tolist()[:3] == [ok_row] * 3 and i[2].tolist()[3:] == [-1] * (k - 3)
    assert _bits_equal(s[2, :1].expand(3), s[2, :3])
    assert int(i[3, 0]) == ok_row                      # the inf row's error is NaN (never ranks) or +inf (after every finite one)
    assert all(int(x) in (41, -1) for x in i[3, 1:]) and bool(torch.isinf(s[3][i[3] == 41]).all())


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("chunk", [128, 1024])
def test_shards_merge_equals_unsharded(engine, chunk):
    """Four row shards, rerank_local on each and codae_topk_merge: the unsharded ids; the errors agree within tolerance, and bit
    for bit at chunk = 128, where every chunk is one 128-row tile on every shard."""
    from codae import _C
    from codae.tool.inference import SwapScorer, shard_rows
    n, S, E, slot, Q, m, k = 3000, 3, 64, 1, 40, 100, 12
    model, _, _ = _model(S, E, engine, 41)
    torch.manual_seed(42)
    cat = (torch.rand(n, E) * 2).to(DEV)
    allow = torch.rand(n, device=DEV) < 0.7
    outfits = torch.rand(Q, S * E, device=DEV)
    cand = torch.randint(-50, n + 50, (Q, m), dtype=torch.int64, device=DEV)
    whole = SwapScorer(model, cat, E, k=k, chunk=chunk, allowed=allow)
    s_ref, i_ref = (t.clone() for t in whole.rerank(outfits, slot, cand))
    parts = []
    for r in range(4):
        lo, nl = shard_rows(n, 4, r)
        sc = SwapScorer(model, cat[lo:lo + nl], E, k=k, row_offset=lo, chunk=chunk, allowed=allow[lo:lo + nl])
        parts.append(tuple(t.clone() for t in sc.rerank_local(outfits, slot, cand)))
    gs = torch.stack([p[0] for p in parts])
    gi = torch.stack([p[1] for p in parts])
    ms, mi = torch.empty_like(s_ref), torch.empty_like(i_ref)
    _C.topk_merge(gs, gi, _C.METRIC_SQERR, ms, mi)
    assert torch.equal(mi, i_ref)
    assert np.allclose(ms.cpu().numpy(), s_ref.cpu().numpy(), rtol=RTOL[engine], atol=1e-6)
    if chunk == 128:
        assert _bits_equal(ms, s_ref)
    assert bool(allow[mi[mi >= 0]].all())


def _guarded(bufs, nbytes, guard=4096):            # 0xff bytes: NaN as float32, -1 as integers
    buf = torch.full((guard + nbytes + guard,), 255, dtype=torch.uint8, device=DEV)
    bufs.append(buf)
    return buf[guard:guard + nbytes]


def test_outputs_stay_in_bounds_and_bad_arguments_are_rejected():
    """pos entries outside [0, Q m) and ids outside the catalog are never dereferenced: their rows are built as zeros and get no
    error; nothing is written outside the guarded buffers; bad shapes / k / NULL return CODAE_EINVAL."""
    from codae import _C
    n, S, E, slot, Q, m, k, guard = 300, 2, 64, 1, 6, 5, 4, 4096
    io = S * E
    torch.manual_seed(51)
    bufs = []
    cat = _guarded(bufs, n * E * 4).view(torch.float32).view(n, E)
    cat.copy_(torch.rand(n, E, device=DEV))
    outfits = _guarded(bufs, Q * io * 4).view(torch.float32).view(Q, io)
    outfits.copy_(torch.rand(Q, io, device=DEV))
    cand = _guarded(bufs, Q * m * 8).view(torch.int64).view(Q, m)
    cand.copy_(torch.randint(0, n, (Q, m), device=DEV))
    cand[1, 2] = n + 10 ** 9
    cand[2, 0] = -(10 ** 9)
    pos = _guarded(bufs, 8 * 8).view(torch.int64)
    pos.copy_(torch.tensor([0, Q * m, -5, 3, 1 * m + 2, 2 * m, 10 ** 12, Q * m - 1], device=DEV))   # valid: 0, 3, Q m - 1
    B = pos.numel()
    x = _guarded(bufs, B * io * 4).view(torch.float32).view(B, io)
    y = _guarded(bufs, B * io * 4).view(torch.float32).view(B, io)
    y.zero_()
    err = _guarded(bufs, Q * m * 4).view(torch.float32)
    out_s = _guarded(bufs, Q * k * 4).view(torch.float32).view(Q, k)
    out_i = _guarded(bufs, Q * k * 8).view(torch.int64).view(Q, k)
    before = [b.clone() for b in bufs]
    _C.swap_build_pairs(outfits, cat, 0, cand, pos, E, slot, io, 1.0, x)
    _C.swap_error_pairs(outfits, cat, 0, cand, pos, E, slot, io, 1.0, y, err)
    _C.swap_pairs_topk(err, cand, k, out_s, out_i)
    torch.cuda.synchronize()
    for bb, b0 in zip(bufs, before):
        assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])
    for b in (1, 2, 4, 5, 6):                                  # invalid pos or id: zero rows
        assert bool((x[b] == 0).all()), b
    written = {0, 3, Q * m - 1}
    assert torch.isnan(err).sum().item() == Q * m - len(written)
    for p in written:
        q, j = divmod(p, m)
        xr = outfits[q].clone()
        xr[slot * E:(slot + 1) * E] = cat[cand[q, j]]
        assert abs(float(err[p]) - float((xr.double() ** 2).sum())) <= 1e-5 * float((xr.double() ** 2).sum())
    assert int((out_i >= 0).sum()) == len(written)
    c, L, P = _C.ctx(DEV), _C.lib(), _C.p
    st = _C.stream()

    def build(**kw):
        a = dict(o=P(outfits), ldo=io, Q=Q, cat=P(cat), cdt=_C.F32, ldc=E, n=n, off=0, cand=P(cand), m=m, pos=P(pos), B=B, E=E,
                 slot=slot, io=io, x=P(x), xdt=_C.F32, ldx=io)
        a.update(kw)
        return L.codae_swap_build_pairs(c, a["o"], a["ldo"], a["Q"], a["cat"], a["cdt"], a["ldc"], a["n"], a["off"], a["cand"], a["m"],
                                        a["pos"], a["B"], a["E"], a["slot"], a["io"], 1.0, a["x"], a["xdt"], a["ldx"], st)

    def error(**kw):
        a = dict(o=P(outfits), Q=Q, m=m, E=E, slot=slot, y=P(y), err=P(err), pos=P(pos))
        a.update(kw)
        return L.codae_swap_error_pairs(c, a["o"], io, a["Q"], P(cat), _C.F32, E, n, 0, P(cand), a["m"], a["pos"], B, a["E"],
                                        a["slot"], io, 1.0, a["y"], io, a["err"], st)

    def topk(**kw):
        a = dict(err=P(err), Q=Q, m=m, k=k, s=P(out_s))
        a.update(kw)
        return L.codae_swap_pairs_topk(c, a["err"], P(cand), a["Q"], a["m"], a["k"], a["s"], P(out_i), st)
    assert build() == _C.OK and error() == _C.OK and topk() == _C.OK
    for kw in (dict(Q=0), dict(m=0), dict(E=0), dict(slot=2), dict(slot=-1), dict(o=None), dict(pos=None), dict(x=None), dict(B=0),
               dict(Q=2 ** 20, m=2 ** 12), dict(xdt=7), dict(ldx=io - 1)):
        assert build(**kw) == _C.EINVAL, kw
    for kw in (dict(Q=0), dict(m=0), dict(E=0), dict(slot=2), dict(y=None), dict(err=None), dict(pos=None)):
        assert error(**kw) == _C.EINVAL, kw
    for kw in (dict(k=0), dict(k=129), dict(Q=0), dict(m=0), dict(err=None), dict(s=None)):
        assert topk(**kw) == _C.EINVAL, kw
    torch.cuda.synchronize()


def test_bad_rerank_inputs_raise():
    from codae.tool.inference import SwapScorer
    n, S, E = 100, 2, 64
    model, _, _ = _model(S, E, "fp32", 1)
    sc = SwapScorer(model, torch.rand(n, E, device=DEV), E, k=3)
    o = torch.rand(4, S * E, device=DEV)
    cnd = torch.zeros(4, 3, dtype=torch.int64, device=DEV)
    for args, match in (((o.double(), cnd), "float32"), ((o[:, 1:], cnd), "shape"), ((o, cnd.int()), "int64"),
                        ((o, cnd[:3]), "shape"), ((o.cpu(), cnd), "device"), ((o, cnd.cpu()), "device")):
        with pytest.raises(RuntimeError, match=match):
            sc.rerank_local(args[0], 0, args[1])


def test_embedding_size_planted_swaps():
    """embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)), bf16 engine, a 1 M-row catalog, Q = 1024 outfits x 100
    listed ids.  The untrained DAE's outputs are small, so rows near zero are near-perfect swaps: three planted per list come
    back first, and the errors match the fp64 oracle."""
    from codae.tool.inference import SwapScorer
    n, S, E, slot, Q, m, k = 1_000_000, 3, 512, 2, 1024, 100, 10
    model, W, b = _model(S, E, "bf16", 61, z=1536, nin=4, nout=4)
    assert len(model.dims) == 10
    g = torch.Generator(device=DEV).manual_seed(62)
    cat = torch.rand((n, E), generator=g, device=DEV) + 0.5
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    cand = torch.randint(300_000, n, (Q, m), generator=g, device=DEV, dtype=torch.int64)
    planted = torch.arange(3 * Q, device=DEV).view(Q, 3) * 97 + 11           # distinct rows, below 300 000: in no random list
    cat[planted.flatten()] = 1e-3 * torch.rand((3 * Q, E), generator=g, device=DEV)
    cols = torch.stack([torch.randperm(m - 1, generator=torch.Generator().manual_seed(q))[:3] for q in range(Q)]).to(DEV)
    cand.scatter_(1, cols, planted)
    cand[:, -1] = -1
    sc = SwapScorer(model, cat, E, k=k)
    s, i = (t.cpu() for t in sc.rerank(outfits, slot, cand))
    pl = planted.cpu()
    for q in range(Q):
        assert set(i[q, :3].tolist()) == set(pl[q].tolist()), q
    check = [0, 1, 500, 1023]
    ref = _oracle_pairs([w.to(DEV) for w in W], [x.to(DEV) for x in b], model.relu, outfits[check], slot, E, cat, cand[check].cpu(), 1.0)
    _check_against_oracle(s[check], i[check], ref, cand[check].cpu(), k, RTOL["bf16"])


def _script(tmp_path, *extra):
    args = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config", os.path.join(PKG, "config", "embedding.yaml"),
            "--synthetic", "3000", "--slot", "1", "--queries", "4", "--exclude_own_item"] + list(extra)
    r = subprocess.run([sys.executable] + args, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_script_rerank_mode(tmp_path):
    M, k = 20, 6
    res = _script(tmp_path, "--mode", "rerank", "--rerank_depth", str(M), "--k", str(k))
    stage1 = _script(tmp_path, "--k", str(M))
    assert res["mode"] == "rerank" and res["depth"] == M and len(res["indices"]) == 4 and len(res["scores"]) == 4
    for q, row in enumerate(res["indices"]):
        assert len(row) == k and q not in row
        assert set(row) <= set(stage1["indices"][q])
        assert res["scores"][q] == sorted(res["scores"][q])
