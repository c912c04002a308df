"""CPU: OutfitCompleter.complete_beam_local / complete_beam against the fake backend of _host_dryrun.py, which type-checks every C-ABI
call (argument count and kinds per codae._C.SIGNATURES).  The spy below stands in for the GPU: codae_complete_beam_error and
codae_complete_error write a deterministic pseudo-error per (outfit, combination, level) at the positions they are given, and
codae_swap_pairs_topk selects by (error, key) as the kernel does.  So the driver's whole search -- the child keys and positions, their
chunking, the levels, outfits finishing early, the decode -- is checked against a plain-Python beam search, together with the launch
sequence per level and engine, the limits, the rank slices and complete's own launch sequence.  Runs in a subprocess because the fake
backend monkeypatches torch."""
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
from codae.tool.inference import shard_rows
calls = []
fake = _C.lib()


def arr(ptr, n, ct):
    return np.ctypeslib.as_array((ct * n).from_address(ptr.value))


def perr(q, c, level):                    # the stand-in partial error of combination c of (global) outfit q at `level`
    return float((q * 7919 + c * 104729 + level * 31) % 97) / 8.0


Q_OFF = [0]                               # global index of the first outfit of the call (rank slices)


class Spy:
    def __getattr__(self, name):
        if name == "codae_linear_engine":          # the fake's engine table plus the fp32-parity engine (csrc/linear.cu)
            return lambda c, dtype, M, N, K: dtype if (dtype in (1, 2) and N >= 32 and K >= 32) else 0
        f = getattr(fake, name)
        def g(*a):
            extra = None
            if name in ("codae_complete_beam_build", "codae_complete_beam_error"):
                Q, W, depth, level, B = a[3], a[13], a[11], a[14], a[16]
                pos = arr(a[15], B, ctypes.c_int64).copy()
                parents = arr(a[12], Q * W, ctypes.c_int64).copy()
                extra = (pos.tolist(), level, W)
                if name == "codae_complete_beam_error":
                    err = arr(a[20], Q * W * depth, ctypes.c_float)
                    for p in pos.tolist():
                        q, t, b = p // (W * depth), (p // depth) % W, p % depth
                        err[p] = perr(Q_OFF[0] + q, int(parents[q * W + t]) + b * depth ** level, level)
            elif name == "codae_complete_error":
                pos = arr(a[13], a[14], ctypes.c_int64).copy()
                extra = pos.tolist()
                err = arr(a[18], a[3] * a[12], ctypes.c_float)
                for p in pos.tolist():
                    if p >= 0:
                        err[p] = perr(Q_OFF[0] + p, 0, -1)
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
            calls.append((name, a, extra))
            return f(*a)
        return g
_C.lib = lambda: Spy()
names = lambda: [n for n, _, _ in calls if not n.endswith("workspace_bytes") and n != "codae_cast_bf16"]
S, E = 4, 32
io = S * E
g = torch.Generator().manual_seed(0)
NCAT = [50, 3, 40, 20]                     # slot 1's catalog is shorter than depth 4
OFFS = [0, 0, 100, 0]
cats = [torch.rand(n, E, generator=g) for n in NCAT]
owned = lambda s, i: i >= 0 and OFFS[s] <= i < OFFS[s] + NCAT[s]


def ref_beam(missing, cand, depth, W, k, q0=0):
    # plain-Python beam search with perr: per outfit [(error, c, ids [S])] of the first k of its last level, or its one m_q = 0 entry
    out = []
    for q in range(missing.shape[0]):
        ms = [s for s in range(S) if missing[q, s]]
        if not ms:
            out.append([(perr(q0 + q, 0, -1), 0, [-1] * S)])
            continue
        beam = [0]
        for j, s in enumerate(ms):
            kids = [(perr(q0 + q, c + b * depth ** j, j), c + b * depth ** j) for c in beam for b in range(depth)
                    if owned(s, int(cand[q, s, b]))]
            sel = sorted(kids)[:W]
            beam = [c for _, c in sel]
        res = []
        for e, c in sel[:k]:
            ids = [-1] * S
            for j, s in enumerate(ms):
                ids[s] = int(cand[q, s, (c // depth ** j) % depth])
            res.append((e, c, ids))
        out.append(res)
    return out


def check(err, ids, want, k):
    for q, res in enumerate(want):
        for e in range(k):
            if e < len(res):
                assert float(err[q, e]) == res[e][0] and ids[q, e].tolist() == res[e][2], (q, e, float(err[q, e]), res[e])
            else:
                assert math.isinf(float(err[q, e])) and bool((ids[q, e] == -1).all()), (q, e)


for dtype, eng in (("bf16", _C.BF16), ("fp32", _C.F32X3), ("fp32_simt", _C.F32)):
    model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype(dtype); model.to(torch.device("cpu"))
    assert model.engine_dtype() == eng, (dtype, model.engine_dtype())
    L = len(model.dims)
    x3 = eng == _C.F32X3
    lin = "codae_linear_fwd_x3" if x3 else "codae_linear_fwd"
    for chunk, Q, depth, W, k in ((16, 13, 4, 3, 2), (250, 30, 3, 5, 5), (7, 5, 2, 1, 1), (1000, 9, 1, 4, 1), (40, 11, 4, 64, 4)):
        comp = OutfitCompleter(model, cats, E, depth=depth, k=k, chunk=chunk, inv_scale=0.5, row_offsets=OFFS)
        outfits = torch.rand(Q, io, generator=g)
        missing = torch.rand(Q, S, generator=g) < 0.5
        missing[0] = False                                  # m_q = 0
        missing[1, :3] = True; missing[1, 3] = False        # m_q = 3, through slot 1's short catalog
        missing[2] = True                                   # m_q = 4
        cand = torch.randint(-2, 60, (Q, S, depth), generator=g)
        cand[:, 2] += 100                                   # slot 2's shard holds global rows 100..139
        cand[3, :, :] = -1                                  # outfit 3: every expansion invalid (if it misses anything)
        m_q = missing.sum(1).tolist()
        m_max, n_full = max(m_q), m_q.count(0)
        calls.clear()
        err, ids = comp.complete_beam_local(outfits, missing, cand, W)
        assert err.shape == (Q, k) and ids.shape == (Q, k, S) and err.dtype == torch.float32 and ids.dtype == torch.int64
        check(err, ids, ref_beam(missing, cand, depth, W, k), k)
        # launch sequence: the m_q = 0 outfits through complete_build / _error, then per level its chunks and one selection
        per = lambda b, e: [b] + (["codae_split_x3"] if x3 else []) + [lin] * L + [e]
        nch = lambda n: (n + chunk - 1) // chunk
        want = (["codae_split_x3"] if x3 else []) + per("codae_complete_build", "codae_complete_error") * nch(n_full)
        levels = []
        for j in range(m_max):
            lv = [e for n, a, e in calls if n == "codae_complete_beam_build" and e[1] == j]
            n_rows = sum(len(e[0]) for e in lv)
            assert [len(e[0]) for e in lv] == [min(chunk, n_rows - i) for i in range(0, n_rows, chunk)], (j, lv)
            levels.append(sum((e[0] for e in lv), []))
            want += per("codae_complete_beam_build", "codae_complete_beam_error") * nch(n_rows) + ["codae_swap_pairs_topk"]
        assert names() == want, (dtype, names(), want)
        assert [e for n, _, e in calls if n == "codae_complete_beam_build"] == [e for n, _, e in calls if n == "codae_complete_beam_error"]
        # child positions of level j: every valid child of the reference beam, ascending, at (q W + t) depth + b
        for j, pos in enumerate(levels):
            exp = []
            for q in range(Q):
                ms = [s for s in range(S) if missing[q, s]]
                if j >= len(ms):
                    continue
                beam = [0]
                for jj in range(j):
                    kids = sorted((perr(q, c + b * depth ** jj, jj), c + b * depth ** jj) for c in beam for b in range(depth)
                                  if owned(ms[jj], int(cand[q, ms[jj], b])))
                    beam = [c for _, c in kids[:W]]
                exp += [(q * W + t) * depth + b for t in range(len(beam)) for b in range(depth) if owned(ms[j], int(cand[q, ms[j], b]))]
            assert pos == exp, (j, pos, exp)
        assert all(a[13] == W and a[11] == depth and a[3:6] == (Q, S, E) and a[17] == 0.5
                   for n, a, _ in calls if n.startswith("codae_complete_beam")), "arguments"
        ce = [e for n, _, e in calls if n == "codae_complete_error"]
        assert sum(ce, []) == [q for q in range(Q) if m_q[q] == 0]
        assert all(a[12] == 1 for n, a, _ in calls if n in ("codae_complete_build", "codae_complete_error"))
        for a in (a for n, a, _ in calls if n == "codae_swap_pairs_topk"):
            assert a[3:6] == (Q, W * depth, W), a
        # complete's own sequence is unchanged by the beam: chunks of build / error and one selection over [Q, depth^m_max]
        if depth ** m_max <= _C.COMPLETE_MAX_COMBOS:
            calls.clear()
            comp.complete_local(outfits, missing, cand)
            n_b = len([1 for n, _, _ in calls if n == "codae_complete_build"])
            assert names() == (["codae_split_x3"] if x3 else []) + per("codae_complete_build", "codae_complete_error") * n_b + [
                "codae_swap_pairs_topk"], names()
            assert not any(n.startswith("codae_complete_beam") for n, _, _ in calls)

# limits raise RuntimeError before any call; depth^m past the exhaustive cap is fine for the beam
model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype("bf16"); model.to(torch.device("cpu"))
comp = OutfitCompleter(model, cats, E, depth=17, k=4)
outfits = torch.rand(5, io, generator=g)
three = torch.zeros(5, S, dtype=torch.bool); three[1, [0, 2, 3]] = True      # 17^3 = 4913 combinations > 4096: beam only
cand = torch.zeros(5, S, 17, dtype=torch.int64)
calls.clear()
comp.complete_beam_local(outfits, three, cand, 4)
assert names().count("codae_swap_pairs_topk") == 3
none = three.clone(); none[3, 1] = True
comp_none = OutfitCompleter(model, [cats[0], None, cats[2], cats[3]], E, depth=17, k=4)
calls.clear()
for c, args, match in ((comp, (outfits, three, 0), "width"), (comp, (outfits, three, 129), "width"),
                       (comp, (outfits, three, 3), "exceeds the beam width"),
                       (comp_none, (outfits, none, 4), "no catalog"),
                       (comp, (outfits.double(), three, 4), "float32"), (comp, (outfits, three.int(), 4), "bool")):
    for fn in (c.complete_beam, lambda o, m, w: c.complete_beam_local(o, m, cand, w)):
        try:
            fn(*args); raise AssertionError("accepted %s" % match)
        except RuntimeError as e:
            assert match in str(e), (match, e)
big = OutfitCompleter(model, cats, E, depth=128, k=4)
nine = torch.zeros(2, S, dtype=torch.bool); nine[0] = True
try:                                                                   # 128^4 = 2^28 is fine; S = 4 caps m_q, so test the key
    big.complete_beam_local(torch.zeros(2, io), nine, torch.zeros(2, S, 128, dtype=torch.int64), 4)
except RuntimeError as e:
    raise AssertionError("refused 128^4 keys: %s" % e)
many = torch.zeros(2 ** 31 // (128 * 16) + 1, S, dtype=torch.bool); many[:, 0] = True
calls.clear()
try:
    big.complete_beam_local(torch.zeros(many.shape[0], io), many, torch.zeros(many.shape[0], S, 16, dtype=torch.int64), 128)
    raise AssertionError("accepted Q W depth > 2**31 - 1")
except RuntimeError as e:
    assert "2**31" in str(e), e
assert not names(), names()
# depth^m_max > 2^62: 128^9 = 2^63 on a 10-slot model
S10 = 10
m10 = EmbeddingDenoisingAutoencoder(S10 * E, 40, E, 2, 2, False); m10.set_compute_dtype("bf16"); m10.to(torch.device("cpu"))
c10 = OutfitCompleter(m10, [torch.rand(5, E)] * S10, E, depth=128, k=1)
miss10 = torch.zeros(1, S10, dtype=torch.bool); miss10[0, :9] = True
try:
    c10.complete_beam_local(torch.zeros(1, S10 * E), miss10, torch.zeros(1, S10, 128, dtype=torch.int64), 1)
    raise AssertionError("accepted 128^9 keys")
except RuntimeError as e:
    assert "2**62" in str(e), e
assert not names(), names()

# complete_beam() on 1..4 ranks: the pool is exchanged once, rank r searches its shard_rows slice, two padded gathers; the slices
# equal the reference beam of those outfits
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
    missing = torch.zeros(Q, S, dtype=torch.bool); missing[:, 1] = True; missing[::2, 3] = True; missing[1::3] = False
    cand = torch.randint(0, 3, (Q, S, 2), generator=g)
    for G in (1, 2, 3, 4):
        covered = []
        per = (Q + G - 1) // G
        for r in range(G):
            dist.get_world_size = lambda group=None: G
            dist.get_rank = lambda group=None: r
            comp = OutfitCompleter(model, cats, E, depth=2, k=2, chunk=5, process_group=object())
            lo, n = shard_rows(Q, G, r)
            Q_OFF[0] = lo
            calls.clear(); gathers.clear(); reduces.clear()
            err, ids = comp.complete_beam(outfits, missing, 3, cand)
            Q_OFF[0] = 0
            assert err.shape == (Q, 2) and ids.shape == (Q, 2, S)
            nm = int(missing.sum())
            assert reduces == [(torch.int32, 2 * nm * 2 + nm * 2 * E, dist.ReduceOp.SUM)], reduces
            assert [x[:2] for x in gathers] == [((G * per, 2), (per, 2)), ((G * per, 2, S), (per, 2, S))], gathers
            b = [a for nm_, a, _ in calls if nm_ in ("codae_complete_beam_build", "codae_complete_build")]
            if n:
                assert b and all(a[1].value == outfits.data_ptr() + lo * io * 4 and a[3] == n for a in b), (lo, n)
                covered += list(range(lo, lo + n))
                check(err[:n], ids[:n], ref_beam(missing[lo:lo + n], cand[lo:lo + n], 2, 3, 2, q0=lo), 2)
            else:
                assert not b
        assert covered == list(range(Q)), (Q, G, covered)
print("BEAM OK")
"""


def test_beam_completion_host_orchestration():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "BEAM OK" in r.stdout
