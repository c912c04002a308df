"""CPU: the filtered complementarity top-k (ComplementarityScorer / SwapScorer with `allowed` / `exclude`) against the fake
backend of _host_dryrun.py, which type-checks every C-ABI call (argument count and kinds per codae._C.SIGNATURES).  Runs in a
subprocess because the fake backend monkeypatches torch."""
import os
import subprocess
import sys

SCRIPT = r"""
import sys, ctypes, torch
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
from codae import _C
from codae.tool.inference import ComplementarityScorer
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
names = lambda: [n for n, _ in calls if not n.endswith("workspace_bytes")]
Q, m = 70, 3
ex = torch.full((Q, m), -1, dtype=torch.int64)
for dtype, metric in ((torch.float32, "sqerr"), (torch.bfloat16, "cosine")):
    sc = ComplementarityScorer(torch.rand(300, 32).to(dtype), 32, metric=metric, k=5, row_offset=7,
                               allowed=torch.rand(300) < 0.5)
    assert sc.allowed.dtype == torch.uint8
    s, i = sc.topk_batched(torch.rand(Q, 32), exclude=ex)
    assert s.shape == (Q, 5) and sc.last_fallbacks == 0
    sc.topk(torch.rand(4, 32), exclude=ex[:4])
assert names().count("codae_score_topk_batched_filtered") == 2 and names().count("codae_score_topk_filtered") == 2, names()
assert "codae_score_topk_batched" not in names() and "codae_score_topk" not in names(), names()
a = dict(calls)["codae_score_topk_filtered"]
assert a[12] is not None and a[13] is not None and a[14] == m, a[12:15]      # allow, exclude, n_exclude
calls.clear()
# exclusions alone; an empty [Q, 0] list is passed as (NULL, 0)
sc = ComplementarityScorer(torch.rand(300, 32), 32, k=5)
sc.topk_local(torch.rand(4, 32), exclude=torch.empty((4, 0), dtype=torch.int64))
a = dict(calls)["codae_score_topk_filtered"]
assert a[12] is None and a[13] is None and a[14] == 0, a[12:15]
calls.clear()
# no filter: the unfiltered names, as before
sc.topk_batched(torch.rand(Q, 32))
sc.topk(torch.rand(4, 32))
assert names() == ["codae_score_topk_batched", "codae_score_topk"], names()
calls.clear()
# fallback of uncertified queries: the sweep gets the same mask and the exclusion rows of those queries
orig = _C.score_topk_batched
def two_uncertified(*a, **kw):
    orig(*a, **kw)
    a[9].fill_(2); a[10][:2] = torch.tensor([4, 9], dtype=torch.int32)
_C.score_topk_batched = two_uncertified
seen = {}
orig_sweep = _C.score_topk
def sweep(*a, **kw):
    seen.update(kw, Q=a[3].shape[0])
    return orig_sweep(*a, **kw)
_C.score_topk = sweep
sc = ComplementarityScorer(torch.rand(300, 32), 32, k=5, allowed=torch.ones(300, dtype=torch.bool))
ex = torch.arange(Q * m, dtype=torch.int64).view(Q, m)
sc.topk_local_batched(torch.rand(Q, 32), exclude=ex)
assert sc.last_fallbacks == 2 and seen["Q"] == 2 and seen["allow"] is sc.allowed
assert torch.equal(seen["exclude"], ex[[4, 9]]), seen["exclude"]
assert names() == ["codae_score_topk_batched_filtered", "codae_score_topk_filtered"], names()
# bad filters raise before any call
for bad in (dict(allowed=torch.ones(299, dtype=torch.bool)), dict(allowed=torch.ones(300, dtype=torch.int32))):
    try:
        ComplementarityScorer(torch.rand(300, 32), 32, k=5, **bad); raise AssertionError(bad)
    except RuntimeError:
        pass
for bad in (torch.zeros(Q, 257, dtype=torch.int64), torch.zeros(Q - 1, 2, dtype=torch.int64), torch.zeros(Q, 2, dtype=torch.int32)):
    try:
        sc.topk_local_batched(torch.rand(Q, 32), exclude=bad); raise AssertionError(bad.shape)
    except RuntimeError:
        pass
print("FILTERED OK")
"""


def test_filtered_topk_issues_well_typed_calls():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "FILTERED OK" in r.stdout
