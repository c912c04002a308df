"""CPU: OutfitCompleter against the fake backend of _host_dryrun.py, which type-checks every C-ABI call (argument count and kinds
per codae._C.SIGNATURES): the launch sequence per chunk for each engine, the built positions and their chunking, the combination
decode, the candidate pool, the rank slices and the limits.  Runs in a subprocess because the fake backend monkeypatches torch.
The int32-SUM pool exchange runs on a gloo world of 2."""
import os
import socket
import subprocess
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import PKG, ROOT

SCRIPT = r"""
import ctypes, itertools, sys, torch
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
import torch.distributed as dist
from codae import _C
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool import OutfitCompleter
from codae.tool.inference import _decode_combinations, shard_rows
calls = []
fake = _C.lib()
class Spy:
    def __getattr__(self, name):
        if name == "codae_linear_engine":          # the fake's engine table plus the fp32-parity engine (csrc/linear.cu)
            return lambda c, dtype, M, N, K: dtype if (dtype in (1, 2) and N >= 32 and K >= 32) else 0
        f = getattr(fake, name)
        def g(*a):
            extra = None
            if name in ("codae_complete_build", "codae_complete_error"):      # the positions, read while the tensor is alive
                extra = list((ctypes.c_int64 * a[14]).from_address(a[13].value))
            calls.append((name, a, extra))
            return f(*a)
        return g
_C.lib = lambda: Spy()
names = lambda: [n for n, _, _ in calls if not n.endswith("workspace_bytes") and n != "codae_cast_bf16"]
S, E = 4, 32
io = S * E
g = torch.Generator().manual_seed(0)
NCAT = [50, 3, 40, 20]                     # slot 1's catalog is shorter than depth 4
cats = [torch.rand(n, E, generator=g) for n in NCAT]


def brute_valid(missing, cand, depth, owned):
    # [(q, c)] of every valid combination, ascending, and its ids [S]
    out = {}
    for q in range(missing.shape[0]):
        ms = [s for s in range(S) if missing[q, s]]
        for c in range(depth ** len(ms)):
            ids = [-1] * S
            ok = True
            for j, s in enumerate(ms):
                i = int(cand[q, s, (c // depth ** j) % depth])
                ok &= owned(s, i)
                ids[s] = i
            if ok:
                out[(q, c)] = ids
    return out


for dtype, eng in (("bf16", _C.BF16), ("fp32", _C.F32X3), ("fp32_simt", _C.F32)):
    model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype(dtype); model.to(torch.device("cpu"))
    assert model.engine_dtype() == eng, (dtype, model.engine_dtype())
    L = len(model.dims)
    x3 = eng == _C.F32X3
    lin = "codae_linear_fwd_x3" if x3 else "codae_linear_fwd"
    for chunk, Q, depth in ((16, 13, 4), (250, 30, 3), (7, 5, 2), (1000, 9, 1)):
        comp = OutfitCompleter(model, cats, E, depth=depth, k=5, chunk=chunk, inv_scale=0.5, row_offsets=[0, 0, 100, 0])
        outfits = torch.rand(Q, io, generator=g)
        missing = torch.rand(Q, S, generator=g) < 0.5
        missing[0] = False                                  # m_q = 0
        missing[1, :3] = True; missing[1, 3] = False        # m_q = 3
        cand = torch.randint(-2, 60, (Q, S, depth), generator=g)
        cand[:, 2] += 100                                   # slot 2's shard holds global rows 100..139
        owned = lambda s, i: i >= 0 and [0, 0, 100, 0][s] <= i < [0, 0, 100, 0][s] + NCAT[s]
        want = brute_valid(missing, cand, depth, owned)
        m_max = int(missing.sum(1).max())
        C = depth ** m_max
        calls.clear()
        err, ids = comp.complete_local(outfits, missing, cand)
        assert err.shape == (Q, 5) and ids.shape == (Q, 5, S) and err.dtype == torch.float32 and ids.dtype == torch.int64
        n_valid = len(want)
        n_chunks = (n_valid + chunk - 1) // chunk
        per_chunk = ["codae_complete_build"] + (["codae_split_x3"] if x3 else []) + [lin] * L + ["codae_complete_error"]
        assert names() == (["codae_split_x3"] if x3 else []) + per_chunk * n_chunks + ["codae_swap_pairs_topk"], (dtype, names())
        builds = [(a, e) for n, a, e in calls if n == "codae_complete_build"]
        errs = [(a, e) for n, a, e in calls if n == "codae_complete_error"]
        # positions: every valid (q, c) once, ascending, in chunks of `chunk`; build and error see the same list
        pos = sum((e for _, e in builds), [])
        assert pos == sorted(q * C + c for q, c in want), (pos, sorted(want))
        assert [len(e) for _, e in builds] == [min(chunk, n_valid - i) for i in range(0, n_valid, chunk)]
        assert [e for _, e in builds] == [e for _, e in errs]
        eng_, acts, stage = comp._dae.buffers()
        dst = acts[0] if stage is None else stage
        for (a, _), (b, _) in zip(builds, errs):
            assert a[1].value == b[1].value and a[2] == io and a[3:6] == (Q, S, E) and a[11:13] == (depth, C), a
            assert a[15] == 0.5 and a[16].value == dst.data_ptr() and a[17] == _C.dt(dst) and a[18] == dst.stride(0), a
            assert b[16].value == acts[-1].data_ptr() and b[17] == acts[-1].stride(0), b
        topk = [a for n, a, _ in calls if n == "codae_swap_pairs_topk"][0]
        assert topk[3:6] == (Q, C, 5), topk
        # the pool: slot-major missing pairs, depth rows each, the owned catalog rows (un-scaled) and zeros elsewhere
        x, miss, cc = comp._inputs(outfits, missing, cand)
        counts, m_max2, C2 = comp._limits(miss, depth)
        assert (m_max2, C2) == (m_max, C) and counts == missing.sum(0).tolist()
        slot_base, pool, pool_id = comp._pool(miss, cc, counts, depth)
        i = 0
        for s in range(S):
            for q in range(Q):
                if not missing[q, s]:
                    assert slot_base[q, s] == -1
                    continue
                assert slot_base[q, s] == i * depth
                for j in range(depth):
                    gid = int(cand[q, s, j])
                    row, rid = pool[i * depth + j], int(pool_id[i * depth + j])
                    if owned(s, gid):
                        assert rid == gid and torch.equal(row, cats[s][gid - [0, 0, 100, 0][s]]), (q, s, j)
                    else:
                        assert rid == -1 and not bool(row.any()), (q, s, j)
                i += 1
        assert pool.shape == (max(1, i * depth), E)
        # decode: the ids of every valid combination; -1 for unused entries
        qs = sorted({q for q, _ in want})
        for q in range(Q):
            cs = [c for qq, c in want if qq == q][:5]
            combo = torch.tensor([cs + [-1] * (5 - len(cs))])
            got = _decode_combinations(combo, slot_base[q:q + 1], pool_id, depth)[0]
            for e, c in enumerate(cs):
                assert got[e].tolist() == want[(q, c)], (q, c, got[e].tolist(), want[(q, c)])
            assert (got[len(cs):] == -1).all()
        # the pool rows of a valid combination are exactly what the build kernel reads: slot_base + digit
        for (q, c), ids_ in want.items():
            ms = [s for s in range(S) if missing[q, s]]
            for j, s in enumerate(ms):
                assert int(pool_id[slot_base[q, s] + (c // depth ** j) % depth]) == ids_[s]

# stage 1: one masked forward (mul_mask), one sweep per missing slot; the [Q, S, depth] lists go where they belong
model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype("bf16"); model.to(torch.device("cpu"))
comp = OutfitCompleter(model, [cats[0], None, cats[2], cats[3]], E, depth=3, k=4, row_offsets=[0, 0, 100, 0])
Q = 6
outfits = torch.rand(Q, io, generator=g)
missing = torch.zeros(Q, S, dtype=torch.bool); missing[:, 0] = True; missing[2:, 3] = True
calls.clear()
cand = comp.candidates(outfits, missing)
assert cand.shape == (Q, S, 3) and cand.dtype == torch.int64
assert names()[:2] == ["codae_mul_mask", "codae_linear_fwd"] and names().count("codae_score_topk") == 2, names()
sweeps = [a for n, a, _ in calls if n == "codae_score_topk"]
assert sweeps[0][3] == 50 and sweeps[0][8] == Q and sweeps[1][3] == 20 and sweeps[1][8] == Q - 2, [(a[3], a[8]) for a in sweeps]
assert sweeps[1][6] == 0 and sweeps[0][11] == 3
assert (cand[:, 1:3] == -1).all() and (cand[:2, 3] == -1).all()

# limits and bad inputs raise RuntimeError before any call
calls.clear()
for kw in (dict(depth=0), dict(depth=129), dict(k=0), dict(k=129), dict(chunk=0), dict(row_offsets=[0, 0])):
    try:
        OutfitCompleter(model, cats, E, **kw); raise AssertionError("accepted %s" % kw)
    except RuntimeError:
        pass
for bad in ([cats[0]] * 3, [cats[0].double()] + cats[1:], [cats[0][:, :E - 1]] + cats[1:]):
    try:
        OutfitCompleter(model, bad, E); raise AssertionError("accepted catalogs")
    except RuntimeError:
        pass
comp = OutfitCompleter(model, [cats[0], None, cats[2], cats[3]], E, depth=17, k=4)
outfits = torch.rand(5, io, generator=g)
missing = torch.zeros(5, S, dtype=torch.bool); missing[0, 0] = True
cand = torch.zeros(5, S, 17, dtype=torch.int64)
three = missing.clone(); three[1, [0, 2, 3]] = True                          # 17^3 = 4913 combinations > 4096
none = missing.clone(); none[3, 1] = True                                    # slot 1 has no catalog
for args, match in (((outfits, three), "combinations"), ((outfits, three, cand), "combinations"), ((outfits, none), "no catalog"),
                    ((outfits.double(), missing), "float32"), ((outfits[:, 1:], missing), "shape"),
                    ((outfits, missing.int()), "bool"), ((outfits, missing[:, :3]), "shape"), ((outfits, missing[:4]), "shape"),
                    ((outfits, missing, cand.int()), "int64"), ((outfits, missing, cand[:, :3]), "shape"),
                    ((outfits, missing, torch.zeros(5, S, 129, dtype=torch.int64)), "shape")):
    for fn in (comp.complete, comp.complete_local) if len(args) == 3 else (comp.complete, comp.candidates):
        try:
            fn(*args); raise AssertionError("accepted %s" % match)
        except RuntimeError as e:
            assert match in str(e), (match, e)
big = OutfitCompleter(model, cats, E, depth=16, k=4)
many = torch.zeros(2 ** 31 // 4096 + 1, S, dtype=torch.bool); many[:, :3] = True    # Q C = (2**19 + 1) 4096 > 2**31 - 1
try:
    big.complete(torch.zeros(many.shape[0], io), many, torch.zeros(many.shape[0], S, 16, dtype=torch.int64))
    raise AssertionError("accepted Q C > 2**31 - 1")
except RuntimeError as e:
    assert "2**31" in str(e), e
assert not names(), names()

# complete() on 1..4 ranks: the pool is exchanged once, rank r runs stage 2 on its shard_rows slice, two padded gathers
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
comp_args = (model, cats, E)
for Q in (1, 2, 7, 10):
    outfits = torch.rand(Q, io, generator=g)
    missing = torch.zeros(Q, S, dtype=torch.bool); missing[:, 1] = True; missing[::2, 3] = True
    cand = torch.randint(0, 3, (Q, S, 2), generator=g)
    for G in (1, 2, 3, 4):
        covered = []
        per = (Q + G - 1) // G
        for r in range(G):
            dist.get_world_size = lambda group=None: G
            dist.get_rank = lambda group=None: r
            comp = OutfitCompleter(*comp_args, depth=2, k=3, chunk=5, process_group=object())
            calls.clear(); gathers.clear(); reduces.clear()
            err, ids = comp.complete(outfits, missing, cand)
            assert err.shape == (Q, 3) and ids.shape == (Q, 3, S)
            nm = int(missing.sum())
            assert reduces == [(torch.int32, 2 * nm * 2 + nm * 2 * E, dist.ReduceOp.SUM)], reduces
            assert [x[:2] for x in gathers] == [((G * per, 3), (per, 3)), ((G * per, 3, S), (per, 3, S))], gathers
            lo, n = shard_rows(Q, G, r)
            b = [a for nm_, a, _ in calls if nm_ == "codae_complete_build"]
            if n:
                assert b and all(a[1].value == outfits.data_ptr() + lo * io * 4 and a[3] == n for a in b), (lo, n)
                covered += list(range(lo, lo + n))
            else:
                assert not b
        assert covered == list(range(Q)), (Q, G, covered)
print("COMPLETE OK")
"""


def test_completion_issues_well_typed_calls():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "COMPLETE OK" in r.stdout


def _exchange_worker(rank, world, port, q):
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from codae.tool.inference import _exchange_pool
        R, E = 12, 5
        g = torch.Generator().manual_seed(1)
        full = torch.randn(R, E, generator=g)
        full[0, 0], full[1, 1], full[2, 2], full[3, 3], full[4, 4] = -0.0, float("nan"), float("inf"), float("-inf"), 0.0
        full[5, :] = float("nan")
        ids = torch.arange(R, dtype=torch.int64) * 1_000_003 + 2 ** 40      # ids above 2**32: both int32 halves carry bits
        owner = torch.tensor([0, 1, 0, 1, 0, 1, 0, 1, -1, 0, 1, -1])        # -1: a row no rank holds
        mine = owner == rank
        pool = torch.where(mine.view(-1, 1), full, 0.0)
        pool_id = torch.where(mine, ids, -1)
        out, out_id = _exchange_pool(pool, pool_id, None)
        held = owner >= 0
        want = torch.where(held.view(-1, 1), full, 0.0)
        assert torch.equal(out.view(torch.int32), want.view(torch.int32)), (out, want)
        assert torch.equal(out_id, torch.where(held, ids, -1)), out_id
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_pool_exchange_on_a_gloo_world_of_two():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_exchange_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == {0: "ok", 1: "ok"}, res
