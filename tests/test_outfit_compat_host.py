"""CPU: CompatibilityScorer.score_local / score against the fake backend of _host_dryrun.py, which type-checks every C-ABI call
(argument count and kinds per codae._C.SIGNATURES), and compatibility_auc against a brute-force pair count.  Runs in a subprocess
because the fake backend monkeypatches torch."""
import os
import subprocess
import sys

import pytest

SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
import torch.distributed as dist
from codae import _C
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool.inference import CompatibilityScorer, shard_rows
calls = []
fake = _C.lib()
class Spy:
    def __getattr__(self, name):
        if name == "codae_linear_engine":          # the fake's engine table plus the fp32-parity engine (csrc/linear.cu)
            return lambda c, dtype, M, N, K: dtype if (dtype in (1, 2) and N >= 32 and K >= 32) else 0
        f = getattr(fake, name)
        def g(*a):
            calls.append((name, a))
            return f(*a)
        return g
_C.lib = lambda: Spy()
names = lambda: [n for n, _ in calls if not n.endswith("workspace_bytes") and n != "codae_cast_bf16"]
S, E = 3, 32
io = S * E
for dtype, eng in (("bf16", _C.BF16), ("fp32", _C.F32X3), ("fp32_simt", _C.F32)):
    model = EmbeddingDenoisingAutoencoder(io, 40, E, 2, 2, False); model.set_compute_dtype(dtype); model.to(torch.device("cpu"))
    assert model.engine_dtype() == eng, (dtype, model.engine_dtype())
    L = len(model.dims)
    x3 = eng == _C.F32X3
    lin = "codae_linear_fwd_x3" if x3 else "codae_linear_fwd"
    for chunk, Q in ((16, 13), (250, 300), (9, 3), (4, 2)):
        sc = CompatibilityScorer(model, E, chunk=chunk)
        per = chunk // S
        outfits = torch.rand(Q, io)
        calls.clear()
        err, score, odd = sc.score_local(outfits)
        assert err.shape == (Q, S) and score.shape == (Q,) and odd.shape == (Q,)
        assert err.dtype == torch.float32 and score.dtype == torch.float32 and odd.dtype == torch.int64
        chunks = [(c0, min(per, Q - c0)) for c0 in range(0, Q, per)]
        per_chunk = ["codae_corrupt_fwd"] * S + (["codae_split_x3"] if x3 else []) + [lin] * L + ["codae_outfit_loo_error"]
        assert names() == (["codae_split_x3"] if x3 else []) + per_chunk * len(chunks), (dtype, chunk, names())
        eng_, acts, stage = sc._dae.buffers()
        assert acts[0].shape[-2] == per * S and (stage is not None) == x3
        dst = acts[0] if stage is None else stage
        cor = [a for n, a in calls if n == "codae_corrupt_fwd"]
        lins = [a for n, a in calls if n == lin]
        loo = [a for n, a in calls if n == "codae_outfit_loo_error"]
        for j, (c0, Bq) in enumerate(chunks):
            for s in range(S):
                a = cor[j * S + s]
                assert a[1].value == outfits.data_ptr() + c0 * io * 4 and a[2] == Bq and a[4] is None and a[5] == Bq, a
                assert a[7] == S and a[8] == s and a[11] == io and a[13] == _C.dt(dst), a
                assert a[12].value == dst.data_ptr() + s * Bq * dst.stride(0) * dst.element_size() and a[14] == dst.stride(0), a
            for l in range(L):
                M = lins[j * L + l][10 if x3 else 8]
                assert M == S * Bq and M % S == 0, (M, Bq)               # chunk rows: whole outfits, slot-major
            a = loo[j]
            assert a[1].value == outfits.data_ptr() + c0 * io * 4 and a[2] == io and a[3:6] == (Bq, S, E), a
            assert a[6].value == acts[-1].data_ptr() and a[7] == acts[-1].stride(0), a
            assert a[8].value == err.data_ptr() + c0 * S * 4 and a[9].value == score.data_ptr() + c0 * 4, a
            assert a[10].value == odd.data_ptr() + c0 * 8, a
# chunk < S is refused
for bad in (dict(chunk=2), dict(chunk=0)):
    try:
        CompatibilityScorer(model, E, **bad); raise AssertionError("accepted %s" % bad)
    except Exception as e:
        assert "chunk" in str(e), e
# bad inputs raise RuntimeError before any call
sc = CompatibilityScorer(model, E, chunk=64)
calls.clear()
outfits = torch.rand(5, io)
for o in (outfits.double(), outfits[:, :-1], outfits[0], outfits[:0], outfits.numpy(), outfits.tolist(), outfits.view(5, S, E)):
    try:
        sc.score_local(o); raise AssertionError("accepted %s" % type(o))
    except RuntimeError:
        pass
assert not names(), names()
# score() on 1..4 ranks: each rank scores its shard_rows slice, every rank gathers three padded tensors, the slices cover Q
gathers = []
def all_gather_into_tensor(out, t, group=None):
    gathers.append((tuple(out.shape), tuple(t.shape), t.dtype))
    out.copy_(t.repeat((out.shape[0] // t.shape[0],) + (1,) * (t.dim() - 1)))
dist.is_available = lambda: True
dist.is_initialized = lambda: True
dist.all_gather_into_tensor = all_gather_into_tensor
for Q in (1, 2, 7, 10):
    outfits = torch.rand(Q, io)
    for G in (1, 2, 3, 4):
        covered = []
        per = (Q + G - 1) // G
        for r in range(G):
            dist.get_world_size = lambda group=None: G
            dist.get_rank = lambda group=None: r
            sc = CompatibilityScorer(model, E, chunk=9, process_group=object())
            calls.clear(); gathers.clear()
            err, score, odd = sc.score(outfits)
            assert err.shape == (Q, S) and score.shape == (Q,) and odd.shape == (Q,)
            assert [g[:2] for g in gathers] == [((G * per, S), (per, S)), ((G * per,), (per,)), ((G * per,), (per,))], gathers
            lo, n = shard_rows(Q, G, r)
            rows = [(int((a[1].value - outfits.data_ptr()) // (io * 4)), a[3]) for nm, a in calls if nm == "codae_outfit_loo_error"]
            if n:
                assert rows[0][0] == lo and sum(b for _, b in rows) == n, (rows, lo, n)
                covered += list(range(lo, lo + n))
            else:
                assert not rows
        assert covered == list(range(Q)), (Q, G, covered)
print("COMPAT OK")
"""


def test_compat_issues_well_typed_calls():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "COMPAT OK" in r.stdout


def _brute_auc(pos, neg):
    import math
    pos = [p for p in pos if not math.isnan(p)]
    neg = [n for n in neg if not math.isnan(n)]
    wins = sum((p < n) + 0.5 * (p == n) for p in pos for n in neg)
    return wins / (len(pos) * len(neg))


@pytest.mark.parametrize("seed", range(6))
def test_compatibility_auc_matches_pair_count(seed):
    import torch
    from codae.tool.inference import compatibility_auc
    g = torch.Generator().manual_seed(seed)
    n_p, n_n = int(torch.randint(1, 60, (1,), generator=g)), int(torch.randint(1, 60, (1,), generator=g))
    pos = torch.randint(0, 12, (n_p,), generator=g).float()        # few distinct values: many ties, within and across the sets
    neg = torch.randint(3, 15, (n_n,), generator=g).float()
    if seed % 2:
        pos[torch.rand(n_p, generator=g) < 0.2] = float("nan")
        neg[torch.rand(n_n, generator=g) < 0.2] = float("nan")
        pos[0], neg[0] = 1.0, 1.0                                  # at least one finite score on each side
    want = _brute_auc(pos.tolist(), neg.tolist())
    assert abs(compatibility_auc(pos, neg) - want) < 1e-12


def test_compatibility_auc_edges():
    import math
    import torch
    from codae.tool.inference import compatibility_auc
    assert compatibility_auc(torch.tensor([1.0, 2.0]), torch.tensor([3.0, 4.0])) == 1.0
    assert compatibility_auc(torch.tensor([3.0, 4.0]), torch.tensor([1.0, 2.0])) == 0.0
    assert compatibility_auc(torch.tensor([2.0]), torch.tensor([2.0])) == 0.5
    assert math.isnan(compatibility_auc(torch.tensor([float("nan")]), torch.tensor([1.0])))
