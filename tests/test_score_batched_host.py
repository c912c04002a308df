"""CPU: ComplementarityScorer.topk_batched / topk_local_batched against the fake backend of _host_dryrun.py, which type-checks
every C-ABI call (argument count and kinds per codae._C.SIGNATURES).  Runs in a subprocess because the fake backend
monkeypatches torch."""
import os
import subprocess
import sys

SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import _host_dryrun                       # installs the fake backend (and runs its own dry run first)
from codae import _C
from codae.tool.inference import ComplementarityScorer
calls = []
fake = _C.lib()
class Spy:
    def __getattr__(self, name):
        calls.append(name)
        return getattr(fake, name)
_C.lib = lambda: Spy()
for dtype, metric in ((torch.float32, "sqerr"), (torch.bfloat16, "cosine")):
    sc = ComplementarityScorer(torch.rand(300, 32).to(dtype), 32, metric=metric, k=5, row_offset=7)
    s, i = sc.topk_batched(torch.rand(70, 32))
    assert s.shape == (70, 5) and i.shape == (70, 5) and sc.last_fallbacks == 0
assert calls.count("codae_score_topk_batched") == 2 and "codae_score_topk" not in calls, calls
calls.clear()
sc = ComplementarityScorer(torch.rand(300, 32), 32, k=65)          # beyond the tensor-core path: the sweep alone
s, i = sc.topk_batched(torch.rand(9, 32))
assert s.shape == (9, 65) and sc.last_fallbacks == 9 and calls.count("codae_score_topk") == 1
assert "codae_score_topk_batched" not in calls, calls
print("BATCHED OK")
"""


def test_topk_batched_issues_well_typed_calls():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", SCRIPT, here], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "BATCHED OK" in r.stdout
