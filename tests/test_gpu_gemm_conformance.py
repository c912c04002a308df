"""GEMM conformance: every launch plan of the three linear contractions on the three engines, exact against an fp64 reference
(tests/_gemm_conformance_cases.py explains why integer operands make the exact answer representable).

The case matrix runs in a child process under a timeout: CODAE_DEBUG_PLAN is read once per process, and a protocol bug in a
persistent kernel must not take the test session with it.  Besides every case being exact, the plan each case logged must be
the one the Python mirror of the plan choice predicts, and together the logged plans must reach every required plan cell."""
import os
import subprocess
import sys
import time

import pytest

import _gemm_conformance_cases as G

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def run_matrix():
    env = {k: v for k, v in os.environ.items() if k not in G.PLAN_KNOBS}
    env["CODAE_DEBUG_PLAN"] = "1"
    t0 = time.time()
    r = subprocess.run([sys.executable, os.path.join(HERE, "_gemm_conformance_cases.py")], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300, env=env)
    return r, time.time() - t0


def parse(out):
    """{case id: (result text, [plan lines])}, {prefetch case: result}, SM count."""
    cases, prefetch, sm, cur, plans = {}, {}, None, None, []
    for line in out.splitlines():
        if line.startswith("SMS "):
            sm = int(line.split()[1])
        elif line.startswith("CASE "):
            cur, plans = line[5:], []
        elif line.startswith("codae plan:") and cur is not None:
            plans.append(line)
        elif line.startswith("RESULT ") and cur is not None and line.startswith("RESULT " + cur + " "):
            cases[cur] = (line[len("RESULT " + cur + " "):], plans)
            cur, plans = None, []
        elif line.startswith("PREFETCH "):
            how, res = line[len("PREFETCH "):].rsplit(" ", 1)
            prefetch[how] = res
    return cases, prefetch, sm


def test_every_gemm_plan_is_exact_and_reached():
    r, secs = run_matrix()
    out = r.stdout
    assert r.returncode == 0 and "DONE" in out, out[-6000:]
    cases, prefetch, sm = parse(out)
    matrix = G.case_matrix(sm)
    failures, plans, wrong_plan = [], {}, []
    for c in matrix:
        assert c["id"] in cases, "case %s did not report" % c["id"]
        res, lines = cases[c["id"]]
        if not res.startswith("ok"):
            failures.append("%s: %s" % (c["id"], res))
        parsed = [G.parse_plan(l) for l in lines]
        parsed = [p for p in parsed if p is not None]
        want = G.expected_plan(sm, c)
        dims = G.gemm_dims(c["op"], c["M"], c["N"], c["K"])
        if len(parsed) != 1 or parsed[0][0] != dims or parsed[0][1] != want:
            wrong_plan.append("%s: logged %s, mirror %s" % (c["id"], lines, want))
        else:
            plans[c["id"]] = parsed[0][1]
    assert not failures, "\n".join(failures)
    assert not wrong_plan, "\n".join(wrong_plan)
    assert prefetch == {"cast same stream": "ok", "adam same stream": "ok", "cast side stream": "ok"}, prefetch
    cov = G.coverage(sm, plans)
    missing = sorted(G.required_cells() - set(cov))
    assert not missing, missing
    # coverage table: cell -> first case that reached it -> its plan line
    print("\n%d cases on %d SMs in %.1f s" % (len(matrix), sm, secs))
    for cell in sorted(G.required_cells()):
        cid = cov[cell][0]
        print("| %s | %s | %s |" % (cell, cid, cases[cid][1][0].replace("codae plan: ", "")))
    for c in matrix:
        if c["random"]:
            print("random-valued %s: %s" % (c["eng"], cases[c["id"]][0]))
