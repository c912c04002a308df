"""CPU: SwapScorer.rerank_local / rerank against the fake backend of _host_dryrun.py, which type-checks every C-ABI call (argument
count and kinds per codae._C.SIGNATURES).  Runs in a subprocess because the fake backend monkeypatches torch."""
import os
import subprocess
import sys

SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
from codae import _C
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool.inference import SwapScorer, shard_rows
calls = []
fake = _C.lib()
class Spy:
    def __getattr__(self, name):
        f = getattr(fake, name)
        def g(*a):
            calls.append((name, a))
            return f(*a)
        return g
_C.lib = lambda: Spy()
names = lambda: [n for n, _ in calls if not n.endswith("workspace_bytes") and n not in ("codae_linear_engine", "codae_cast_bf16")]
S, E, n, k = 3, 32, 300, 5
for dtype in ("fp32", "bf16"):
    model = EmbeddingDenoisingAutoencoder(S * E, 40, E, 2, 2, False); model.set_compute_dtype(dtype); model.to(torch.device("cpu"))
    L = len(model.dims)
    cat = torch.rand(n, E)
    torch.manual_seed(0)
    Q, m = 7, 40
    cand = torch.randint(-20, n + 20, (Q, m), dtype=torch.int64)      # padding and ids outside the catalog
    cand[3] = -1                                                       # an all-padding list
    allow = torch.rand(n) < 0.6
    outfits = torch.rand(Q, S * E)
    # four row shards: their positions are disjoint, ascending and cover exactly the valid, allowed, non-padding entries
    seen = []
    for rank in range(4):
        lo, nl = shard_rows(n, 4, rank)
        sw = SwapScorer(model, cat[lo:lo + nl], E, k=k, row_offset=lo, chunk=16, allowed=allow[lo:lo + nl])
        pos = sw._owned_positions(cand)
        assert pos.dtype == torch.int64 and bool((pos[1:] > pos[:-1]).all())
        seen.append(pos)
        calls.clear()
        s, i = sw.rerank_local(outfits, 1, cand)
        assert s.shape == (Q, k) and i.shape == (Q, k) and s.dtype == torch.float32 and i.dtype == torch.int64
        chunks = (pos.numel() + 15) // 16
        x3 = sw._buffers()[2] is not None          # fp32-parity engine: built in the fp32 stage, then split into planes
        per_chunk = ["codae_swap_build_pairs"] + (["codae_split_x3"] if x3 else []) + \
                    ["codae_linear_fwd_x3" if x3 else "codae_linear_fwd"] * L + ["codae_swap_error_pairs"]
        assert names() == per_chunk * chunks + ["codae_swap_pairs_topk"], names()
        b = [a for nm, a in calls if nm == "codae_swap_build_pairs"]
        assert [a[12] for a in b] == [min(16, pos.numel() - c0) for c0 in range(0, pos.numel(), 16)], b     # B per chunk
        assert all(a[3] == Q and a[7] == nl and a[8] == lo and a[10] == m for a in b), b
        t = dict(calls)["codae_swap_pairs_topk"]
        assert t[3:6] == (Q, m, k), t
    allp = torch.cat(seen)
    flat = cand.view(-1)
    valid = (flat >= 0) & (flat < n)
    want = torch.nonzero(valid & allow[flat.clamp(0, n - 1)]).view(-1)
    assert allp.numel() == allp.unique().numel() and torch.equal(allp.sort().values, want)
    # bad inputs raise before any call
    sw = SwapScorer(model, cat, E, k=k, chunk=16)
    calls.clear()
    bad = [(outfits.double(), cand), (outfits[:, :-1], cand), (outfits[0], cand), (outfits, cand.int()), (outfits, cand[:-1]),
           (outfits, cand[:, :0]), (outfits, cand.view(-1)), (outfits.numpy(), cand), (outfits, cand.tolist())]
    for o, c in bad:
        try:
            sw.rerank_local(o, 1, c); raise AssertionError("accepted %s" % type(o))
        except RuntimeError:
            pass
    big = torch.empty((1, 2 ** 31), dtype=torch.int64).expand(2, 2 ** 31)   # Q m > 2**31 - 1 (no storage for it is needed)
    try:
        sw.rerank_local(outfits[:2], 1, big); raise AssertionError("accepted Q m > 2**31 - 1")
    except RuntimeError:
        pass
    assert not names(), names()
    # topk_local issues the call sequence it issued before rerank existed
    sw = SwapScorer(model, cat, E, k=k, chunk=128)
    calls.clear()
    sw.topk_local(outfits[0], 1)
    x3 = sw._buffers()[2] is not None
    per_chunk = ["codae_swap_build"] + (["codae_split_x3"] if x3 else []) + \
                ["codae_linear_fwd_x3" if x3 else "codae_linear_fwd"] * L + ["codae_swap_error_topk"]
    assert names() == per_chunk * 3 + ["codae_topk_merge"], names()
    rs, ri = sw.rerank(outfits, 1, cand)
    assert rs.shape == (Q, k)
print("RERANK OK")
"""


def test_rerank_issues_well_typed_calls():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "RERANK OK" in r.stdout
