"""GPU tests of the batched complementarity top-k (codae_score_topk_batched, ComplementarityScorer.topk_local_batched /
topk_batched): tensor-core proposals certified against the row sweep must return exactly what the sweep returns."""
import math

import numpy as np
import pytest
import torch

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


def _both(cat, E, q, metric, k, inv_scale=0.5, row_offset=1000):
    from codae.tool.inference import ComplementarityScorer
    sc = ComplementarityScorer(cat.to(DEV).contiguous(), E, metric=metric, k=k, inv_scale=inv_scale, row_offset=row_offset)
    qd = q.to(DEV)
    s_ref, i_ref = (t.clone() for t in sc.topk_local(qd))
    s, i = sc.topk_local_batched(qd)
    return sc, s.clone(), i.clone(), s_ref, i_ref


GRID = [  # n, E, Q, k, metric, bf16, specials
    (7, 16, 1, 10, "sqerr", False, False), (7, 64, 129, 1, "cosine", True, False),
    (5000, 16, 63, 10, "sqerr", True, True), (5000, 64, 128, 64, "cosine", False, True),
    (5000, 512, 1000, 10, "sqerr", False, False), (5000, 512, 129, 10, "cosine", True, False),
    (5000, 1536, 63, 1, "sqerr", True, False), (5000, 4096, 129, 64, "sqerr", False, False),
    (300_001, 512, 1000, 10, "sqerr", True, True), (300_001, 512, 128, 64, "cosine", True, True),
    (300_001, 64, 1000, 10, "cosine", False, False), (300_001, 1536, 129, 10, "sqerr", False, True),
    (300_001, 4096, 63, 1, "cosine", True, False), (300_001, 4096, 1, 10, "sqerr", True, False),
]


@pytest.mark.parametrize("n,E,Q,k,metric,bf16,specials", GRID)
def test_batched_equals_sweep(n, E, Q, k, metric, bf16, specials):
    cat = _catalog(n, E, bf16, n + E + k, specials)
    q = _queries(cat, Q, E, Q + k)
    sc, s, i, s_ref, i_ref = _both(cat, E, q, metric, k)
    assert torch.equal(i, i_ref)
    assert torch.equal(s.view(torch.int32), s_ref.view(torch.int32))          # bit for bit (NaN-safe)
    if n > 1000 and not specials:
        assert sc.last_fallbacks == 0


@pytest.mark.parametrize("n,E,Q,k,metric,bf16", [(5000, 512, 130, 10, "sqerr", False), (5000, 64, 64, 7, "cosine", True),
                                                 (7, 512, 3, 10, "sqerr", False)])
def test_batched_matches_oracle(n, E, Q, k, metric, bf16):
    from oracle import codae_oracle as O
    cat = _catalog(n, E, bf16, n + E + k)
    q = _queries(cat, Q, E, Q + k)
    _, s, i, _, _ = _both(cat, E, q, metric, k)
    s, i = s.cpu(), i.cpu()
    for qi in range(0, Q, 13):
        scores = O.score_candidates(cat.float(), q[qi], metric, inv_scale=0.5)
        ws, wi = O.topk(scores, k, metric, row_offset=1000)
        m = min(k, n)
        assert i[qi, :m].tolist() == wi.tolist(), (qi, i[qi, :m], wi)
        assert torch.all(i[qi, m:] == -1)
        assert np.allclose(s[qi, :m].numpy(), ws.numpy(), rtol=2e-5, atol=1e-6)


def test_uncertifiable_queries_fall_back():
    """More than k' identical copies at the k-th place: the bound cannot separate them from the rows left out, so exactly
    those queries fall back to the sweep -- and the results are still the sweep's."""
    from codae.tool.inference import ComplementarityScorer
    n, E, k, Q = 20000, 64, 10, 200
    kp = min(2 * k + 32, 128)
    torch.manual_seed(3)
    cat = torch.rand(n, E)
    q = torch.rand(Q, E)
    tied = [5, 77, 150]
    row = 100
    for qi in tied:
        for j in range(k - 1):                              # k - 1 clear winners
            cat[row] = q[qi] + 1e-3 * (j + 1); row += 1
        for _ in range(kp + 8):                             # then more than k' identical rows at the k-th place
            cat[row] = q[qi] + 2e-2; row += 1
    sc = ComplementarityScorer(cat.to(DEV), E, "sqerr", k)
    s_ref, i_ref = (t.clone() for t in sc.topk_local(q.to(DEV)))
    s, i = sc.topk_local_batched(q.to(DEV))
    assert sc.last_fallbacks == len(tied)
    assert torch.equal(i, i_ref) and torch.equal(s, s_ref)
    sc2 = ComplementarityScorer(torch.rand(n, E).to(DEV), E, "sqerr", k)
    sc2.topk_local_batched(q.to(DEV))
    assert sc2.last_fallbacks == 0


@pytest.mark.parametrize("metric,bf16", [("sqerr", True), ("sqerr", False), ("cosine", True), ("cosine", False)])
def test_proposal_bound_holds(metric, bf16):
    """The proposals' keys (documented at the start of the workspace) bound the exact scores: |a - s| <= delta, i.e.
    key <= s <= key + 2 delta for SQERR (mirrored for COSINE), with s in fp64."""
    from codae import _C
    from codae.tool.inference import ComplementarityScorer
    n, E, Q, k, s_inv = 40000, 512, 130, 10, 0.5
    torch.manual_seed(9)
    cat = torch.rand(n, E)
    if bf16:
        cat = cat.to(torch.bfloat16)
    q = torch.rand(Q, E)
    sc = ComplementarityScorer(cat.to(DEV), E, metric, k, inv_scale=s_inv)
    sc.topk_local_batched(q.to(DEV))
    ws = sc._workspace_batched(Q)[0]
    kp = min(2 * k + 32, 128)
    key = ws[:Q * kp * 4].view(torch.float32).view(Q, kp).cpu().double()
    off = (Q * kp * 4 + 255) // 256 * 256
    idx = ws[off:off + Q * kp * 8].view(torch.int64).view(Q, kp).cpu()
    assert bool((idx >= 0).all())
    c = cat.double()[idx]                                   # [Q, kp, E]
    qd = q.double()[:, None, :]
    P = 2 if bf16 else 3
    c_rel = (2 ** -14 + (P * math.ceil(E / 16) + 8) * 2 ** -21 + (E / 32 + 16) * 2 ** -21) * (1 + 2 ** -10)
    if metric == "sqerr":
        s = ((qd - c * s_inv) ** 2).sum(-1)
        delta = c_rel * ((qd ** 2).sum(-1) + s_inv ** 2 * (c ** 2).sum(-1))
        assert bool((key <= s).all()) and bool((s <= key + 2 * delta * (1 + 1e-3)).all())
    else:
        s = (c * qd).sum(-1) / ((c ** 2).sum(-1) * (qd ** 2).sum(-1)).sqrt().clamp_min(1e-8)
        delta = c_rel * (1 + s.abs())
        assert bool((key >= s).all()) and bool((s >= key - 2 * delta * (1 + 1e-3)).all())


def test_shards_merge_equals_unsharded():
    from codae import _C
    from codae.tool.inference import ComplementarityScorer, shard_rows
    n, E, k, G, Q = 30011, 512, 10, 4, 300
    torch.manual_seed(0)
    cat = torch.randn(n, E).abs().to(DEV)
    q = torch.randn(Q, E).abs().to(DEV)
    full = ComplementarityScorer(cat, E, "sqerr", k)
    ref_s, ref_i = (t.clone() for t in full.topk_local(q))
    b_s, b_i = (t.clone() for t in full.topk_local_batched(q))
    ps, pi = [], []
    for r in range(G):
        lo, c = shard_rows(n, G, r)
        s, i = ComplementarityScorer(cat[lo:lo + c], E, "sqerr", k, row_offset=lo).topk_local_batched(q)
        ps.append(s.clone()); pi.append(i.clone())
    ms, mi = torch.empty_like(ref_s), torch.empty_like(ref_i)
    _C.topk_merge(torch.stack(ps), torch.stack(pi), _C.METRIC_SQERR, ms, mi)
    assert torch.equal(mi, ref_i) and torch.equal(ms, ref_s)
    assert torch.equal(b_i, ref_i) and torch.equal(b_s, ref_s)


def test_full_size_planted_near_copies():
    """10 M x 512 bf16 catalog, Q = 1024, k = 10: planted near-copies come back in order, every list equals the sweep's,
    and a second call returns the same bits."""
    from codae.tool.inference import ComplementarityScorer
    n, E, k, Q = 10_000_000, 512, 10, 1024
    g = torch.Generator(device=DEV).manual_seed(11)
    cat = torch.rand((n, E), generator=g, device=DEV).to(torch.bfloat16)
    q = torch.rand((Q, E), generator=g, device=DEV)
    planted = {}
    for qi in (0, 17, 500, 1023):
        rows = torch.randint(0, n, (k,), generator=g, device=DEV).tolist()
        for j, r in enumerate(rows):
            cat[r] = (q[qi] + 2e-2 * (j + 1)).to(cat.dtype)
        planted[qi] = rows
    sc = ComplementarityScorer(cat, E, "sqerr", k)
    s, i = (t.clone() for t in sc.topk_local_batched(q))
    assert sc.last_fallbacks == 0
    for qi, rows in planted.items():
        assert i[qi].tolist() == rows
    s_ref, i_ref = sc.topk_local(q)
    assert torch.equal(i, i_ref) and torch.equal(s, s_ref)
    s2, i2 = sc.topk_local_batched(q)
    assert torch.equal(s2, s) and torch.equal(i2, i)


@pytest.mark.parametrize("bf16", [False, True])
def test_outputs_and_workspace_bounds(bf16):
    """Outputs and workspace in NaN-filled guarded allocations: nothing outside them is written."""
    from codae import _C
    n, E, Q, k, guard = 9000, 64, 200, 10, 4096
    torch.manual_seed(1)
    cat = torch.rand(n, E, device=DEV)
    if bf16:
        cat = cat.to(torch.bfloat16)
    q = torch.rand(Q, E, device=DEV)
    nws = _C.score_topk_batched_workspace(cat, E, Q, k).numel()
    bufs = []

    def guarded(nbytes):                        # 0xff bytes: NaN as float32, -1 as integers
        buf = torch.full((guard + nbytes + guard,), 255, dtype=torch.uint8, device=DEV)
        bufs.append(buf)
        return buf[guard:guard + nbytes]
    ws = guarded(nws)
    s = guarded(Q * k * 4).view(torch.float32).view(Q, k)
    i = guarded(Q * k * 8).view(torch.int64).view(Q, k)
    cnt = guarded(4).view(torch.int32)
    unc = guarded(Q * 4).view(torch.int32)
    before = [b.clone() for b in bufs]
    _C.score_topk_batched(cat, E, 0, q, 1.0, _C.METRIC_SQERR, k, s, i, cnt, unc, ws)
    torch.cuda.synchronize()
    for b, b0 in zip(bufs, before):
        assert torch.equal(b[:guard], b0[:guard]) and torch.equal(b[-guard:], b0[-guard:])
    assert int(cnt.view(torch.int32)[0]) == 0
    assert not torch.isnan(s).any()


def test_rejects_out_of_range_k():
    from codae import _C
    cat = torch.rand(100, 64, device=DEV)
    q = torch.rand(4, 64, device=DEV)
    ws = _C.score_topk_batched_workspace(cat, 64, 4, 64)
    s, i = torch.empty(4, 65, device=DEV), torch.empty(4, 65, dtype=torch.int64, device=DEV)
    cnt, unc = torch.zeros(1, dtype=torch.int32, device=DEV), torch.empty(4, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match="outside"):
        _C.score_topk_batched(cat, 64, 0, q, 1.0, _C.METRIC_SQERR, 65, s, i, cnt, unc, ws)
