"""CPU: OutfitCompleter.revise_candidates / revise_local / revise against the fake backend of _host_dryrun.py, which type-checks every
C-ABI call (argument count and kinds per codae._C.SIGNATURES).  The spy below stands in for the GPU: codae_revise_error writes a
deterministic pseudo-error per (outfit, grid column) at the positions it is given, and codae_swap_pairs_topk selects by (error, key)
as the kernel does.  So the driver's whole stage 2 -- the grid positions, their chunking, the pool, the ranking, the cut at the base
row and the decode of keys into (slot, id) -- is checked against a plain-Python restatement, together with the launch sequence per
engine, stage 1's leave-one-slot-out queries and exclusions, the limits, the rank slices, and complete's and CompatibilityScorer's own
launch sequences.  Runs in a subprocess because the fake backend monkeypatches torch."""
import os
import subprocess
import sys

SCRIPT = r"""
import ctypes, math, sys, torch
import numpy as np
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
import torch.distributed as dist
from codae import _C
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool import OutfitCompleter
from codae.tool.inference import CompatibilityScorer, ComplementarityScorer, shard_rows
calls = []
fake = _C.lib()


def arr(ptr, n, ct):
    return np.ctypeslib.as_array((ct * n).from_address(ptr.value))


def perr(q, col):                         # the stand-in swap error of grid column col of (global) outfit q; column 0 is the base
    return float((q * 7919 + col * 104729) % 97) / 8.0 + (2.0 if col == 0 else 0.0)


Q_OFF = [0]                               # global index of the first outfit of the call (rank slices)


class Spy:
    def __getattr__(self, name):
        if name == "codae_linear_engine":          # the fake's engine table plus the fp32-parity engine (csrc/linear.cu)
            return lambda c, dtype, M, N, K: dtype if (dtype in (1, 2) and N >= 32 and K >= 32) else 0
        f = getattr(fake, name)
        def g(*a):
            extra = None
            if name in ("codae_revise_build", "codae_revise_error"):
                Q, S, depth, B = a[3], a[4], a[11], a[13]
                pos = arr(a[12], B, ctypes.c_int64).copy()
                R = a[9]
                extra = (pos.tolist(), arr(a[6], Q * S, ctypes.c_int64).copy(), arr(a[10], R, ctypes.c_int64).copy(),
                         arr(a[7], R * a[8], ctypes.c_float).copy().reshape(R, a[8]))
                if name == "codae_revise_error":
                    G = 1 + S * depth
                    err = arr(a[17], Q * G, ctypes.c_float)
                    for p in pos.tolist():
                        err[p] = perr(Q_OFF[0] + p // G, p % G)
            elif name == "codae_swap_pairs_topk":
                Q, m, k = a[3], a[4], a[5]
                err, key = arr(a[1], Q * m, ctypes.c_float), arr(a[2], Q * m, ctypes.c_int64)
                os_, oi = arr(a[6], Q * k, ctypes.c_float), arr(a[7], Q * k, ctypes.c_int64)
                for q in range(Q):
                    lst = sorted((float(err[q * m + i]), int(key[q * m + i])) for i in range(m)
                                 if key[q * m + i] >= 0 and not math.isnan(err[q * m + i]))[:k]
                    lst += [(math.inf, -1)] * (k - len(lst))
                    for e, (s, i) in enumerate(lst):
                        os_[q * k + e], oi[q * k + e] = s, i
                extra = key.copy().reshape(Q, m)
            calls.append((name, a, extra))
            return f(*a)
        return g
_C.lib = lambda: Spy()
names = lambda: [n for n, _, _ in calls if not n.endswith("workspace_bytes") and n != "codae_cast_bf16"]
S, E = 4, 32
io = S * E
g = torch.Generator().manual_seed(0)
NCAT = [50, 3, 40, 20]
OFFS = [0, 0, 100, 0]
cats = [torch.rand(n, E, generator=g) for n in NCAT]
owned = lambda s, i: i >= 0 and OFFS[s] <= i < OFFS[s] + NCAT[s]


def ref_revise(cand, depth, k, has_cat, q0=0):
    # plain-Python stage 2 with perr: per outfit (base, [(error, slot, id)] of the first k swaps below base)
    out = []
    for q in range(cand.shape[0]):
        base = perr(q0 + q, 0)
        swaps = []
        for s in range(S):
            if not has_cat[s] or not any(int(i) >= 0 for i in cand[q, s]):
                continue
            for c in range(depth):
                if owned(s, int(cand[q, s, c])):
                    swaps.append((perr(q0 + q, 1 + s * depth + c), s * depth + c, s, int(cand[q, s, c])))
        swaps.sort()
        out.append((base, [(e, s, i) for e, _, s, i in swaps if e < base][:k]))
    return out


def check(res, want, k):
    base, err, slot, ids = res
    for q, (b, lst) in enumerate(want):
        assert float(base[q]) == b, (q, float(base[q]), b)
        for e in range(k):
            got = (float(err[q, e]), int(slot[q, e]), int(ids[q, e]))
            assert got == (lst[e] if e < len(lst) else (math.inf, -1, -1)), (q, e, got, lst)


def positions(cand, depth, has_cat):
    G = 1 + S * depth
    exp = []
    for q in range(cand.shape[0]):
        exp.append(q * G)
        for s in range(S):
            if has_cat[s] and any(int(i) >= 0 for i in cand[q, s]):
                exp += [q * G + 1 + s * depth + c for c in range(depth) if owned(s, int(cand[q, s, c]))]
    return exp


for dtype, eng in (("bf16", _C.BF16), ("fp32", _C.F32X3), ("fp32_simt", _C.F32)):
    model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype(dtype); model.to(torch.device("cpu"))
    assert model.engine_dtype() == eng, (dtype, model.engine_dtype())
    L = len(model.dims)
    x3 = eng == _C.F32X3
    lin = "codae_linear_fwd_x3" if x3 else "codae_linear_fwd"
    per = lambda b, e: [b] + (["codae_split_x3"] if x3 else []) + [lin] * L + [e]
    for chunk, Q, depth, k, none_slot in ((16, 13, 4, 3, None), (250, 30, 3, 20, 3), (7, 5, 2, 1, None), (1000, 9, 1, 4, 0),
                                          (3, 4, 4, 128, None)):
        cs = [None if s == none_slot else c for s, c in enumerate(cats)]
        has_cat = [c is not None for c in cs]
        comp = OutfitCompleter(model, cs, E, depth=depth, k=k, chunk=chunk, inv_scale=0.5, row_offsets=OFFS)
        outfits = torch.rand(Q, io, generator=g)
        cand = torch.randint(-2, 60, (Q, S, depth), generator=g)
        cand[:, 2] += 100                                   # slot 2's shard holds global rows 100..139
        cand[1, :, :] = -1                                  # outfit 1: nothing revised, its base alone
        cand[2, 0, :] = -1                                  # outfit 2: slot 0 not revised
        calls.clear()
        res = comp.revise_local(outfits, cand)
        base, err, slot, ids = res
        assert base.shape == (Q,) and err.shape == (Q, k) and slot.shape == (Q, k) and ids.shape == (Q, k)
        assert base.dtype == err.dtype == torch.float32 and slot.dtype == ids.dtype == torch.int64
        check(res, ref_revise(cand, depth, k, has_cat), k)
        # launch sequence: the grid's chunks, then one selection over [Q, 1 + S depth]
        bl = [e for n, a, e in calls if n == "codae_revise_build"]
        n_rows = sum(len(e[0]) for e in bl)
        assert [len(e[0]) for e in bl] == [min(chunk, n_rows - i) for i in range(0, n_rows, chunk)], [len(e[0]) for e in bl]
        assert names() == (["codae_split_x3"] if x3 else []) + per("codae_revise_build", "codae_revise_error") * len(bl) + [
            "codae_swap_pairs_topk"], (dtype, names())
        assert [e[0] for n, _, e in calls if n == "codae_revise_build"] == [e[0] for n, _, e in calls if n == "codae_revise_error"]
        # positions: the base row and every held swap of every outfit, ascending
        assert sum((e[0] for e in bl), []) == positions(cand, depth, has_cat)
        G = 1 + S * depth
        assert all(a[3:6] == (Q, S, E) and a[11] == depth and a[14] == 0.5 for n, a, _ in calls if n.startswith("codae_revise")), "args"
        tk = [(a, e) for n, a, e in calls if n == "codae_swap_pairs_topk"]
        assert len(tk) == 1 and tk[0][0][3:6] == (Q, G, k), tk
        key = tk[0][1]                                      # s depth + c for held swaps, -1 for the base row and the rest
        assert (key[:, 0] == -1).all() and sorted(q * G + 1 + int(v) for q in range(Q) for v in key[q] if v >= 0) == [
            p for p in positions(cand, depth, has_cat) if p % G]
        # the pool: one block of depth rows per revised (outfit, slot) pair, slot-major; rows outside the shards and padding are -1
        _, slot_base, pool_id, pool = bl[0]
        slot_base = slot_base.reshape(Q, S)
        revised = [(q, s) for s in range(S) for q in range(Q) if has_cat[s] and any(int(i) >= 0 for i in cand[q, s])]
        assert sorted(int(v) for v in slot_base.reshape(-1) if v >= 0) == [i * depth for i in range(len(revised))]
        for i, (q, s) in enumerate(revised):
            assert slot_base[q, s] == i * depth
            for c in range(depth):
                gid = int(cand[q, s, c])
                assert pool_id[i * depth + c] == (gid if owned(s, gid) else -1)
                if owned(s, gid):
                    assert np.array_equal(pool[i * depth + c], cats[s][gid - OFFS[s]].numpy())
        assert all(slot_base[q, s] < 0 for q in range(Q) for s in range(S) if (q, s) not in revised)
        # complete's and CompatibilityScorer's own launch sequences are unchanged
        missing = torch.zeros(Q, S, dtype=torch.bool); missing[:, 2] = True
        calls.clear()
        comp.complete_local(outfits, missing, cand)
        n_b = len([1 for n, _, _ in calls if n == "codae_complete_build"])
        assert n_b and names() == (["codae_split_x3"] if x3 else []) + per("codae_complete_build", "codae_complete_error") * n_b + [
            "codae_swap_pairs_topk"], names()
        cc = max(chunk, S)
        sc = CompatibilityScorer(model, E, chunk=cc)
        calls.clear()
        sc.score_local(outfits)
        n_c = (Q + cc // S - 1) // (cc // S)
        assert names() == (["codae_split_x3"] if x3 else []) + (["codae_corrupt_fwd"] * S + (["codae_split_x3"] if x3 else []) +
                                                               [lin] * L + ["codae_outfit_loo_error"]) * n_c, names()

        # stage 1: the leave-one-slot-out pass, then one top-k per slot with a catalog over the outfits that do not keep it, on
        # query rows y[s Bq + i, s E:(s + 1) E] of each chunk and with exclude[q, s]; from TC_MIN_Q outfits up, topk_batched
        comp.revise_candidates(outfits)                     # makes the leave-one-slot-out scorer; it shares the GEMM buffers
        assert (comp._compat._dae is comp._dae) == (chunk >= S)
        eng_, acts, stage = comp._compat._dae.buffers()
        Y = torch.arange(acts[-1].numel(), dtype=torch.float32).view(acts[-1].shape)
        acts[-1].copy_(Y)                                   # the fake GEMMs leave it as it is: every chunk reads this pattern
        seen = {}
        for s, sc_ in enumerate(comp._scorers):
            if sc_ is None:
                continue
            def rec(query, exclude=None, s=s, how="topk"):
                seen[s] = (how, query.clone(), None if exclude is None else exclude.clone())
                n = query.shape[0]
                return torch.zeros(n, depth), torch.arange(n * depth, dtype=torch.int64).view(n, depth) + 1000 * s
            sc_.topk = rec
            sc_.topk_batched = lambda q_, e_=None, s=s, rec=rec: rec(q_, e_, s, "batched")
        for Qs in (Q, 70):
            seen.clear()
            o = torch.rand(Qs, io, generator=g)
            keep = torch.rand(Qs, S, generator=g) < 0.3
            keep[0] = True
            ex = torch.randint(-1, 60, (Qs, S, 3), generator=g)
            calls.clear()
            got = comp.revise_candidates(o, keep, ex)
            nl = names()
            chunk_o = max(chunk, S) // S
            n_c = (Qs + chunk_o - 1) // chunk_o
            assert nl == (["codae_split_x3"] if x3 else []) + (["codae_corrupt_fwd"] * S + (["codae_split_x3"] if x3 else []) +
                                                               [lin] * L) * n_c, nl
            assert got.shape == (Qs, S, depth)
            for s in range(S):
                rows = [q for q in range(Qs) if not keep[q, s]]
                if not has_cat[s] or not rows:
                    assert s not in seen and bool((got[:, s] == -1).all()), s
                    continue
                how, qry, exs = seen[s]
                assert how == ("batched" if len(rows) >= ComplementarityScorer.TC_MIN_Q else "topk"), (s, how)
                assert torch.equal(exs, ex[rows, s])
                for j, q in enumerate(rows):
                    c0 = q // chunk_o * chunk_o
                    Bq = min(chunk_o, Qs - c0)
                    assert torch.equal(qry[j], Y[s * Bq + q - c0, s * E:(s + 1) * E]), (s, q)
                    assert torch.equal(got[q, s], torch.arange(j * depth, (j + 1) * depth) + 1000 * s)
                assert all(bool((got[q, s] == -1).all()) for q in range(Qs) if keep[q, s])
        # without keep no outfit is left out and nothing synchronises in stage 1
        seen.clear()
        comp.revise_candidates(o)
        assert all(seen[s][1].shape[0] == 70 and seen[s][2] is None for s in seen) and len(seen) == sum(has_cat)

# revise() with candidates: keep masks them; the result is revise_local's
model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype("bf16"); model.to(torch.device("cpu"))
comp = OutfitCompleter(model, cats, E, depth=3, k=5, chunk=11, row_offsets=OFFS)
outfits = torch.rand(8, io, generator=g)
cand = torch.randint(0, 60, (8, S, 3), generator=g); cand[:, 2] += 100
keep = torch.rand(8, S, generator=g) < 0.5
check(comp.revise(outfits, keep=keep, candidates=cand), ref_revise(torch.where(keep.unsqueeze(2), -1, cand), 3, 5, [True] * S), 5)

# limits raise RuntimeError before any call
calls.clear()
o = torch.rand(5, io, generator=g)
c3 = torch.zeros(5, S, 3, dtype=torch.int64)
bad = [(dict(keep=torch.zeros(5, S, dtype=torch.int32)), "bool"), (dict(keep=torch.zeros(5, S - 1, dtype=torch.bool)), "shape"),
       (dict(exclude=torch.zeros(5, S, 257, dtype=torch.int64)), "exclude"), (dict(exclude=torch.zeros(5, S, 0, dtype=torch.int64)), "exclude"),
       (dict(exclude=torch.zeros(5, S, 2)), "int64"), (dict(exclude=torch.zeros(5, 2, 2, dtype=torch.int64)), "exclude"),
       (dict(candidates=torch.zeros(5, S, 129, dtype=torch.int64)), "candidates"), (dict(candidates=c3.int()), "int64")]
for kw, match in bad:
    for fn in (comp.revise, lambda x, **kw: comp.revise_candidates(x, kw.get("keep"), kw.get("exclude"))
               if "candidates" not in kw else comp.revise_local(x, kw["candidates"])):
        try:
            fn(o, **kw); raise AssertionError("accepted %s" % kw)
        except RuntimeError as e:
            assert match in str(e), (match, e)
for x_ in (o.double(), o[:, :-1]):
    for fn in (lambda: comp.revise(x_), lambda: comp.revise_local(x_, c3), lambda: comp.revise_candidates(x_)):
        try:
            fn(); raise AssertionError("accepted bad outfits")
        except RuntimeError:
            pass
try:
    comp.revise_local(o, None); raise AssertionError("accepted no candidates")
except RuntimeError as e:
    assert "candidates" in str(e)
S64 = 64                                                   # Q (1 + S depth) > 2**31 - 1 at 64 slots x depth 128
m64 = EmbeddingDenoisingAutoencoder(S64, 40, 1, 2, 2, False); m64.set_compute_dtype("bf16"); m64.to(torch.device("cpu"))
c64 = OutfitCompleter(m64, [torch.rand(5, 1)] * S64, 1, depth=128, k=1)
Qb = (2 ** 31 - 1) // (1 + S64 * 128) + 1
big = torch.zeros(Qb, S64)
for fn in (lambda: c64.revise(big), lambda: c64.revise_candidates(big)):
    try:
        fn(); raise AssertionError("accepted Q (1 + S depth) > 2**31 - 1")
    except RuntimeError as e:
        assert "2**31" in str(e), e
assert not names(), names()

# revise() on 1..4 ranks: the pool is exchanged once, rank r scores its shard_rows slice, four padded gathers; the slices equal the
# reference of those outfits
gathers, reduces = [], []
def all_gather_into_tensor(out, t, group=None):
    gathers.append((tuple(out.shape), tuple(t.shape), t.dtype))
    out.copy_(t.repeat((out.shape[0] // t.shape[0],) + (1,) * (t.dim() - 1)))
def all_reduce(t, op=None, group=None):
    reduces.append((t.dtype, t.numel(), op))
dist.is_available = lambda: True
dist.is_initialized = lambda: True
dist.all_gather_into_tensor = all_gather_into_tensor
dist.all_reduce = all_reduce
for Q in (1, 2, 7, 10):
    outfits = torch.rand(Q, io, generator=g)
    cand = torch.randint(0, 3, (Q, S, 2), generator=g)
    cand[:, 2] += 100
    cand[::3, 1] = -1
    nm = sum(1 for q in range(Q) for s in range(S) if (cand[q, s] >= 0).any())
    for G in (1, 2, 3, 4):
        covered = []
        per = (Q + G - 1) // G
        for r in range(G):
            dist.get_world_size = lambda group=None: G
            dist.get_rank = lambda group=None: r
            comp = OutfitCompleter(model, cats, E, depth=2, k=2, chunk=5, row_offsets=OFFS, process_group=object())
            lo, n = shard_rows(Q, G, r)
            Q_OFF[0] = lo
            calls.clear(); gathers.clear(); reduces.clear()
            res = comp.revise(outfits, candidates=cand)
            Q_OFF[0] = 0
            assert [t.shape for t in res] == [(Q,), (Q, 2), (Q, 2), (Q, 2)]
            assert reduces == [(torch.int32, 2 * nm * 2 + nm * 2 * E, dist.ReduceOp.SUM)], reduces
            assert [x[:2] for x in gathers] == [((G * per,), (per,))] + [((G * per, 2), (per, 2))] * 3, gathers
            b = [a for nm_, a, _ in calls if nm_ == "codae_revise_build"]
            if n:
                assert b and all(a[1].value == outfits.data_ptr() + lo * io * 4 and a[3] == n for a in b), (lo, n)
                covered += list(range(lo, lo + n))
                check([t[:n] for t in res], ref_revise(cand[lo:lo + n], 2, 2, [True] * S, q0=lo), 2)
            else:
                assert not b
        assert covered == list(range(Q)), (Q, G, covered)
print("REVISE OK")
"""


def test_revision_host_orchestration():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "REVISE OK" in r.stdout
