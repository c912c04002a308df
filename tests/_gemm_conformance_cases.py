"""GEMM conformance cases: every launch plan of codae_linear_fwd / _dgrad / _wgrad on the three engines (bf16 tcgen05,
fp32-parity tcgen05, FFMA), checked exactly against an fp64 reference.

Operands are small integers (entries in [-3, 3], bias in [-8, 8], one row in eight of the bf16-output cases in [-30, 30] so that
bf16 outputs really round), so every product and every partial sum is an integer below 2^24: fp32 accumulation is exact in any
summation order, f32 outputs must equal the fp64 product and bf16 outputs its round-to-nearest-even bf16 value.  For the
fp32-parity engine the three operand planes are built by hand (hi = i 2^8, mid = j 2^4, lo = l, |i|, |j|, |l| <= 3) and the
reference is the sum of the six products the engine keeps (hh, hm, mh, mm, hl, lh): every partial sum is a multiple of 2^8 whose
magnitude stays below 9 (2^16 + 2^13 + 3 2^8) K < 2^32 for K <= 6400, so it is again exact in fp32.  Values are compared, so the
sign of a zero is not.  Output buffers have guard rows and padding columns holding a canary that must survive the call; input
padding and guard rows hold NaN, which any read of them would spread into the result.

Two halves:
  * a pure-Python mirror of the plan choice (pick_bn / make_plan / launch in csrc/gemm_tcgen05.cu, launch in csrc/gemm_simt.cu)
    that generates shapes reaching every required plan cell for a given SM count.  tests/test_gemm_conformance_host.py checks
    the coverage without a GPU for 148 and 132 SMs;
  * the runner, `python tests/_gemm_conformance_cases.py`, which runs the case matrix on cuda:0 (CODAE_DEBUG_PLAN=1 must be set:
    the library reads it once) and prints `CASE <id>`, the library's `codae plan:` line and `RESULT <id> ok|FAIL <why>` per case.
    tests/test_gpu_gemm_conformance.py runs it in a child process under a timeout, requires every result to be ok and every
    logged plan to be the one the mirror predicts, so a heuristic change that moves a case off its cell fails instead of
    silently dropping coverage.
"""
import os
import re
import sys
import zlib

BM, BK = 128, 64
X3_CHUNK_KB = 8                      # csrc/gemm_tcgen05.cu: x3_chunk_kb() default
OPTIONS = ("SPLITK", "PDL", "PERSISTENT", "WEIGHT_PREFETCH", "TMA_STORE", "TMA_STORE_PERSISTENT", "CTA_PAIR")
# environment knobs that change plans: the runner removes them so that the library's defaults (and the mirror's) hold
PLAN_KNOBS = ("CODAE_X3_CHUNK_KB", "CODAE_X3_BN", "CODAE_DGRAD_BN", "CODAE_WGRAD_BN", "CODAE_DGRAD_MAXSPLIT", "CODAE_GROUP_M",
              "CODAE_TMA_STORE", "CODAE_TMA_STORE_PERSISTENT", "CODAE_CTA_PAIR")
CANARY = 0.3                         # no integer result equals it, in f32 or in bf16


def cdiv(a, b):
    return (a + b - 1) // b


# ---- mirror of the plan choice ---------------------------------------------------------------------------------------------

def gemm_dims(op, M, N, K):
    """(rows, cols, contraction) of the GEMM behind a linear call with batch M, N outputs and K inputs."""
    return {"fwd": (M, N, K), "dgrad": (M, K, N), "wgrad": (N, K, M)}[op]


def linear_dims(op, gM, gN, gK):
    """Inverse of gemm_dims: (M, N, K) of the linear call whose GEMM is gM x gN x gK."""
    return {"fwd": (gM, gN, gK), "dgrad": (gM, gK, gN), "wgrad": (gK, gM, gN)}[op]


def pick_bn(sm, op, planes, gM, gN):
    tiles_m = cdiv(gM, BM)
    t256, t128 = tiles_m * cdiv(gN, 256), tiles_m * cdiv(gN, 128)
    if planes == 1 and t256 >= sm and gN >= 256:
        return 256
    if t128 >= sm and gN >= 128:
        return 128
    if op == "dgrad" and gN >= 128 and tiles_m == 1:
        return 128
    return 64


def plan_tc(sm, case, opts):
    """The plan csrc/gemm_tcgen05.cu logs for this case.  fp32-parity split-K assumes that every cluster of the launch is
    resident at once (the library shrinks the cluster otherwise), which holds for the few-tile shapes used here."""
    planes = 3 if case["eng"] == "x3" else 1
    gM, gN, gK = gemm_dims(case["op"], case["M"], case["N"], case["K"])
    bn = pick_bn(sm, case["op"], planes, gM, gN)
    gx, gy = cdiv(gN, bn), cdiv(gM, BM)
    tiles, total_kb = gx * gy, cdiv(gK, BK)
    nsplit = 1
    if opts["SPLITK"] and 2 * tiles <= sm and total_kb >= 8:
        want = min(sm // tiles, total_kb // 2, 8)
        if want > 1:
            nsplit = cdiv(total_kb, cdiv(total_kb, want))
    out = case["out"]
    staged = nsplit > 1 or (out == "f32" and tiles <= 2 * sm)
    if planes == 1 and nsplit == 1 and not staged and opts["PERSISTENT"] and tiles > 2 * sm:
        unit = 8 if out == "bf16" else 4
        tma = int(bool(opts["TMA_STORE_PERSISTENT"]) and (gN & ~(unit - 1)) > 0 and case["ldc"] % unit == 0)
        return dict(kind="tc", bn=bn, persistent=1, pair=int(bn == 256 and bool(opts["CTA_PAIR"]) and sm >= 2), tma_store=tma)
    plain = not (case["bias"] or case["relu"] or case["mask"])
    tma = int(bool(opts["TMA_STORE"]) and staged and nsplit == 1 and out == "f32" and plain and case["ldc"] % 4 == 0)
    chunked = int(planes == 3 and cdiv(total_kb, nsplit) > X3_CHUNK_KB)
    return dict(kind="tc", bn=bn, np=planes, gx=gx, gy=gy, nsplit=nsplit, staged=int(staged), tma_store=tma, chunked=chunked,
                persistent=0, pair=0)


def plan_simt(sm, case, opts):
    gM, gN, gK = gemm_dims(case["op"], case["M"], case["N"], case["K"])
    ctas64 = cdiv(gM, 64) * cdiv(gN, 64)
    if ctas64 >= 2 * sm:
        return dict(kind="simt", tile=64, split=1)
    if opts["SPLITK"] and gK >= 256 and gM * gN >= 64 * 64:
        return dict(kind="simt", tile=64, split=max(1, min(sm // ctas64, 8, gK // 128)))
    return dict(kind="simt", tile=32, split=1)


def expected_plan(sm, case):
    """The mirror's plan for a case, under the options its call runs with."""
    opts = {o: 0 if o in case["run_off"] else 1 for o in OPTIONS}
    return plan_simt(sm, case, opts) if case["eng"] == "f32" else plan_tc(sm, case, opts)


_RE_SINGLE = re.compile(r"codae plan: M=(\d+) N=(\d+) K=(\d+) BN=(\d+) NP=(\d+) grid (\d+) x (\d+) x (\d+) stages \d+ smem \d+ "
                        r"tmem \d+ staged (\d) tma_store (\d) chunked (\d)")
_RE_PERSISTENT = re.compile(r"codae plan: M=(\d+) N=(\d+) K=(\d+) BN=(\d+) persistent pair (\d) tma_store (\d) ctas \d+")
_RE_SIMT = re.compile(r"codae plan: simt M=(\d+) N=(\d+) K=(\d+) EPI=\d tile (\d+) split (\d+)")


def parse_plan(line):
    """(GEMM dims, plan dict as plan_tc / plan_simt return it) of a `codae plan:` line, or None."""
    m = _RE_SINGLE.search(line)
    if m:
        v = [int(x) for x in m.groups()]
        return tuple(v[0:3]), dict(kind="tc", bn=v[3], np=v[4], gx=v[5], gy=v[6], nsplit=v[7], staged=v[8], tma_store=v[9],
                                   chunked=v[10], persistent=0, pair=0)
    m = _RE_PERSISTENT.search(line)
    if m:
        v = [int(x) for x in m.groups()]
        return tuple(v[0:3]), dict(kind="tc", bn=v[3], persistent=1, pair=v[4], tma_store=v[5])
    m = _RE_SIMT.search(line)
    if m:
        v = [int(x) for x in m.groups()]
        return tuple(v[0:3]), dict(kind="simt", tile=v[3], split=v[4])
    return None


# ---- plan cells ------------------------------------------------------------------------------------------------------------

def cells_of(sm, case, plan):
    """Names of the plan cells one case reaches under `plan` (the mirror's prediction or the logged plan)."""
    eng, op, out = case["eng"], case["op"], case["out"]
    gM, gN, gK = gemm_dims(op, case["M"], case["N"], case["K"])
    tag = "%s %s" % (eng, op)
    cells = set()
    if case["check_off"]:
        cells.add("options all off" if len(case["check_off"]) == len(OPTIONS) else "options %s off" % "+".join(case["check_off"]))
    if case["random"]:
        cells.add("%s random-valued" % tag)
    if eng == "f32":
        epi = {"fwd": "bias+relu" if case["bias"] else "plain", "dgrad": "mask" if case["mask"] else "plain", "wgrad": "db"}[op]
        cells.add("%s %s %s" % (tag, "split-K" if plan["split"] > 1 else "tile%d" % plan["tile"], epi))
        return cells
    cells.add("%s BN%d" % (tag, plan["bn"]))
    if plan["persistent"]:
        kind = "pair" if plan["pair"] else "single"
        cells.add("%s persistent %s tma_store %d %s" % (tag, kind, plan["tma_store"], out))
        family = "persistent " + kind
        if plan["pair"] and 0 < gM % 256 <= 128:
            cells.add("%s tail pair peer without rows" % tag)
    else:
        family = "split-K" if plan["nsplit"] > 1 else ("staged" if plan["staged"] else "direct")
        if plan["nsplit"] > 1:
            cells.add("%s split-K %s" % (tag, out))
        if plan["chunked"]:
            cells.add("%s chunked%s" % (tag, " split-K" if plan["nsplit"] > 1 else ""))
        if plan["staged"] and plan["nsplit"] == 1:
            cells.add("%s single-pass staged %s tma_store %d" % (tag, out, plan["tma_store"]))
        if not plan["staged"]:
            cells.add("%s direct %s" % (tag, out))
        if op == "dgrad" and plan["bn"] == 128 and gM <= BM and cdiv(gN, 128) < sm:
            cells.add("%s BN128 one-row-tile rule" % tag)
    cells.add("%s out %s" % (tag, out))
    if case["mask"]:
        cells.add("%s mask %s" % (tag, out))
    if case["sq"]:
        cells.add("%s sum-of-squares %s" % (tag, family))
    if case["db"]:
        cells.add("%s column sums" % tag)
    if gM % BM:
        cells.add("%s tail M%%128" % tag)
    if out == "bf16" and gN % 8:
        cells.add("%s tail N%%8 bf16" % tag)
    if out == "f32" and gN % 4:
        cells.add("%s tail N%%4 f32" % tag)
    if gK < 64:
        cells.add("%s tail K<64" % tag)
    if gK % 64:
        cells.add("%s tail K%%64" % tag)
    if gK % 64 == 1:
        cells.add("%s tail K=64n+1" % tag)
    if case["pad"]:
        cells.add("%s pitch > width" % tag)
    return cells


def required_cells():
    """Every plan cell the suite must reach (tests/test_gpu_gemm_conformance.py checks the logged plans against it)."""
    req = set()
    for op in ("fwd", "dgrad", "wgrad"):
        t = "bf16 " + op
        outs = ("f32",) if op == "wgrad" else ("f32", "bf16")
        req |= {t + " BN64", t + " BN128", t + " BN256", t + " split-K f32", t + " single-pass staged f32 tma_store 1",
                t + " single-pass staged f32 tma_store 0", t + " tail M%128", t + " tail pair peer without rows", t + " tail N%4 f32",
                t + " tail K<64", t + " tail K%64", t + " tail K=64n+1", t + " pitch > width"}
        req |= {"%s persistent %s tma_store %d %s" % (t, kind, tma, o) for kind in ("single", "pair") for tma in (0, 1) for o in outs}
        if op != "wgrad":
            req |= {t + " split-K bf16", t + " direct bf16", t + " tail N%8 bf16"}
        t = "x3 " + op
        req |= {t + " BN64", t + " BN128", t + " split-K f32", t + " chunked", t + " chunked split-K", t + " out f32",
                t + " tail M%128", t + " tail K%64", t + " pitch > width"}
        if op != "wgrad":
            req |= {t + " out x3", t + " split-K x3"}
        t = "f32 " + op
        epis = {"fwd": ("bias+relu", "plain"), "dgrad": ("mask", "plain"), "wgrad": ("db",)}[op]
        req |= {"%s %s %s" % (t, path, e) for path in ("tile64", "split-K", "tile32") for e in epis}
    req |= {"bf16 dgrad BN128 one-row-tile rule", "bf16 dgrad mask f32", "bf16 dgrad mask bf16", "x3 dgrad mask f32",
            "x3 dgrad mask x3", "bf16 wgrad column sums"}
    req |= {"bf16 wgrad sum-of-squares " + f for f in ("split-K", "staged", "direct", "persistent single", "persistent pair")}
    req |= {"x3 wgrad sum-of-squares " + f for f in ("split-K", "staged")}
    req |= {"options %s off" % o for o in OPTIONS} | {"options all off"}
    req |= {"%s fwd random-valued" % e for e in ("bf16", "x3", "f32")}
    return req


# ---- the case matrix -------------------------------------------------------------------------------------------------------

def make_case(eng, op, M, N, K, out="f32", bias=False, relu=False, mask=False, sq=False, db=False, pad=True, run_off=(),
              check_off=(), random=False):
    """One linear call.  run_off: options switched off for the call; check_off: the subset that is an 'options off' check
    (the rest is how the case reaches its cell, e.g. CTA_PAIR off for the single-CTA BN = 256 persistent kernel)."""
    gN = gemm_dims(op, M, N, K)[1]
    run_off = tuple(sorted(set(run_off) | set(check_off), key=OPTIONS.index))
    c = dict(eng=eng, op=op, M=M, N=N, K=K, out=out, bias=bias, relu=relu, mask=mask, sq=sq, db=db, pad=pad, random=random,
             run_off=run_off, check_off=tuple(sorted(check_off, key=OPTIONS.index)),
             ldc=cdiv(gN, 8) * 8 + 8 if pad else gN)
    assert pad or gN % 8 == 0
    flags = "".join("+" + s for s, f in (("bias", bias), ("relu", relu), ("mask", mask), ("sq", sq), ("db", db), ("random", random),
                                         ("nopad", not pad)) if f)
    c["id"] = "%s-%s-%dx%dx%d-%s%s%s" % (eng, op, M, N, K, out, flags, "".join(" %s=0" % o for o in run_off))
    return c


def family(eng, gM, gN, gK, ops=("fwd", "dgrad", "wgrad"), outs=None, sq=True, run_off=()):
    """The three contractions (or `ops`) whose GEMM is gM x gN x gK, with each output type and fused epilogue."""
    outs = outs or {"bf16": ("f32", "bf16"), "x3": ("f32", "x3"), "f32": ("f32",)}[eng]
    cs = []
    for op in ops:
        M, N, K = linear_dims(op, gM, gN, gK)
        if op == "wgrad":
            cs.append(make_case(eng, op, M, N, K, "f32", sq=sq and eng != "f32", db=eng == "f32", run_off=run_off))
            if eng == "bf16":
                cs.append(make_case(eng, op, M, N, K, "f32", db=True, run_off=run_off))
            continue
        for out in outs:
            if op == "fwd":
                cs.append(make_case(eng, op, M, N, K, out, bias=eng != "x3", relu=True, run_off=run_off))
            else:
                cs.append(make_case(eng, op, M, N, K, out, mask=True, run_off=run_off))
        if eng != "x3":         # the f32 output without a fused epilogue: the single-pass bulk store, the FFMA plain path
            cs.append(make_case(eng, op, M, N, K, "f32", run_off=run_off))
    return cs


def shapes(sm):
    """GEMM shapes (rows, cols, contraction) of the plan families for `sm` SMs."""
    tm128 = cdiv(sm, 3) + 1                          # 128-row tiles with t128 >= SMs > t256 at 384 columns
    Mp = 33 * BM - 28                                # 33 row tiles, M % 256 = 100: the last CTA pair's peer has no rows
    return dict(
        bn64=(300, 331, 72), k40=(200, 333, 40), k193=(130, 197, 193),
        split=(128, 1536, 1536), split_ragged=(100, 1000, 1100), split_wgrad=(128, 256, 1024),
        bn128=(tm128 * BM - 21, 384, 72), bn256=(cdiv(3 * sm, 4) * BM - 37, 509, 72),
        pers64=(BM * sm + 100, 99, 72), pers256=(Mp, 256 * (cdiv(2 * sm + 1, cdiv(Mp, BM)) + 1) - 53, 72),
        x3_split=(128, 256, 1536), x3_chunk_split=(100, 200, 4600), x3_chunk=((cdiv(sm, 2) + 4) * BM - 28, 128, 1100),
        x3_bn128=(tm128 * BM + 40, 384, 72),
        f32_tile64=(64 * cdiv(2 * sm, 19) - 23, 1200, 72), f32_split=(100, 200, 1000), f32_tile32=(50, 70, 90))


def case_matrix(sm):
    s = shapes(sm)
    cs = []
    # bf16 engine.  BN 64 single pass (direct bf16, staged f32 with / without the bulk store); N % 8 != 0; K < 64; K = 64 n + 1
    for key in ("bn64", "k40", "k193", "split", "split_ragged", "bn128", "bn256"):
        cs += family("bf16", *s[key])
    cs.append(make_case("bf16", "fwd", 256, 256, 64, "f32", pad=False))
    cs.append(make_case("bf16", "wgrad", *linear_dims("wgrad", *s["split_wgrad"]), sq=True))
    # persistent kernel: BN 64 single CTA; BN 256 as CTA pairs and single CTA; bulk-store epilogue on and off
    for key, pair_offs in (("pers64", ((),)), ("pers256", ((), ("CTA_PAIR",)))):
        for po in pair_offs:
            for to in ((), ("TMA_STORE_PERSISTENT",)):
                cs += [c for c in family("bf16", *s[key], run_off=po + to) if not c["db"]]
    # fp32-parity engine
    cs += family("x3", *s["bn64"])
    cs += family("x3", *s["x3_split"])
    cs += family("x3", *s["x3_chunk_split"], outs=("f32",), sq=False)
    cs += family("x3", *s["x3_chunk"], outs=("f32",), sq=False)
    cs += family("x3", *s["x3_bn128"], outs=("f32",), sq=False)
    # FFMA engine: 64 x 64 tiles (>= 2 per SM), cluster split-K, 32 x 32 tiles
    for key in ("f32_tile64", "f32_split", "f32_tile32"):
        cs += family("f32", *s[key])
    # options: one representative case per plan family, each option off alone, then all of them off
    reps = [make_case("bf16", "fwd", *s["split"], "bf16", bias=True, relu=True),
            make_case("bf16", "wgrad", *linear_dims("wgrad", *s["bn64"]), sq=True),
            make_case("bf16", "fwd", *s["bn64"], "bf16", bias=True, relu=True),
            make_case("bf16", "dgrad", *linear_dims("dgrad", *s["pers256"]), "bf16", mask=True),
            make_case("bf16", "wgrad", *linear_dims("wgrad", *s["pers256"]), sq=True),
            make_case("bf16", "fwd", *s["pers64"], "f32"),
            make_case("x3", "fwd", *s["x3_chunk_split"], "f32", relu=True),
            make_case("f32", "fwd", *s["f32_split"], bias=True, relu=True)]
    by_id = {c["id"]: c for c in cs}
    for r in reps:
        for off in [(o,) for o in OPTIONS] + [OPTIONS]:
            c = make_case(r["eng"], r["op"], r["M"], r["N"], r["K"], r["out"], r["bias"], r["relu"], r["mask"], r["sq"], r["db"],
                          r["pad"], check_off=off)
            if c["id"] in by_id:          # the same call already reaches a plan cell with this option off
                by_id[c["id"]]["check_off"] = c["check_off"]
            else:
                cs.append(c)
                by_id[c["id"]] = c
    # one random-valued case per engine (elementwise error bound)
    # (six tiles: the fp32-parity split-K cluster is resident as the mirror assumes)
    cs += [make_case(e, "fwd", 128, 331, 1000, "f32", random=True) for e in ("bf16", "x3", "f32")]
    ids = [c["id"] for c in cs]
    assert len(ids) == len(set(ids)), [i for i in ids if ids.count(i) > 1]
    return cs


def coverage(sm, plans=None):
    """{cell: [case ids]} of the matrix at `sm` SMs, under the logged `plans` ({case id: plan}) or the mirror's."""
    cov = {}
    for c in case_matrix(sm):
        plan = plans[c["id"]] if plans is not None else expected_plan(sm, c)
        for cell in cells_of(sm, c, plan):
            cov.setdefault(cell, []).append(c["id"])
    return cov


# ---- the runner (cuda:0) ---------------------------------------------------------------------------------------------------

# Random-valued cases (128 x 331 x 1000, normal operands): |got - ref| <= c sum_k |a_ik| |b_kj| elementwise, ref the fp64 product of
# the same operands.  Worst ratios measured on an NVIDIA B200 (1000 W limit) at 300 x 331 x 1000: 4.2e-8 (bf16), 3.4e-8 (x3),
# 1.1e-7 (FFMA); c is about four times that.
RANDOM_BOUND = {"bf16": 2e-7, "x3": 2e-7, "f32": 5e-7}


def _run():
    import torch
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "..", "mui-deepautoencoder_b200"))
    from codae import _C as C

    dev = torch.device("cuda", 0)
    C.ctx(dev)
    sm = int(C.lib().codae_ctx_sm_count(C.ctx(dev)))
    bf = torch.bfloat16
    opt_ids = {o: getattr(C, "OPT_" + o) for o in OPTIONS}
    gen = torch.Generator(device=dev)

    def ints(shape, r):
        return torch.randint(-r, r + 1, shape, generator=gen, device=dev).double()

    def mask_values(shape):
        # {-2, -1, -0.0, +0.0, 1, 2}: the mask keeps x > 0, so both zeros must clear
        lut = torch.tensor([-2.0, -1.0, -0.0, 0.0, 1.0, 2.0], dtype=torch.float64, device=dev)
        return lut[torch.randint(0, 6, shape, generator=gen, device=dev)]

    def buffer(rows, cols, dtype, fill, planes=0, pad=True):
        """[rows + 2, pitch] (or [3, rows + 2, pitch]) filled with `fill`; returns (buffer, view of the rows x cols matrix)."""
        ld = cdiv(cols, 8) * 8 + 8 if pad else cols
        shape = (rows + 2, ld) if not planes else (3, rows + 2, ld)
        b = torch.full(shape, fill, dtype=dtype, device=dev)
        return b, (b[:rows, :cols] if not planes else b[:, :rows, :cols])

    def operand(vals, eng, planes=None, pad=True):
        """Device operand holding the double matrix `vals` (or the three planes `planes`), NaN in padding and guard rows."""
        rows, cols = vals.shape
        if eng == "x3":
            b, v = buffer(rows, cols, bf, float("nan"), planes=3, pad=pad)
            for i in range(3):
                v[i].copy_(planes[i].to(bf))
            return v
        b, v = buffer(rows, cols, bf if eng == "bf16" else torch.float32, float("nan"), pad=pad)
        v.copy_(vals)
        return v

    def x3_planes(shape, sq):
        # hi = i 2^8, mid = j 2^4, lo = l, |i|, |j|, |l| <= 3.  A sum-of-squares case needs results whose squares, 32 to a
        # chunk, stay below 2^24: there hi = 2 i, mid = j, lo = l with |i|, |j|, |l| <= 1 (the engine contracts whatever
        # planes it is given, and the six-product reference is exact for any of them)
        if sq:
            return [ints(shape, 1) * 2.0, ints(shape, 1), ints(shape, 1)]
        return [ints(shape, 3) * 256.0, ints(shape, 3) * 16.0, ints(shape, 3)]

    def mm6(a, b, f):
        """Sum of the six plane products the fp32-parity engine keeps."""
        ah, am, al = a
        bh, bm, bl = b
        return f(ah, bh) + f(ah, bm) + f(am, bh) + f(am, bm) + f(ah, bl) + f(al, bh)

    def check_canary(buf, rows, cols, planes):
        b = buf.float()
        if planes:
            return all(check_canary(buf[i], rows, cols, 0) for i in range(3))
        want = torch.tensor(CANARY, dtype=buf.dtype).float().item()
        return bool((b[:rows, cols:] == want).all()) and bool((b[rows:] == want).all())

    def run_case(c):
        eng, op, out, M, N, K = c["eng"], c["op"], c["out"], c["M"], c["N"], c["K"]
        dtype = {"bf16": C.BF16, "x3": C.F32X3, "f32": C.F32}[eng]
        r = 2 if c["sq"] else 3
        hot = out == "bf16"
        # operand values (double); A is the operand whose rows are the GEMM rows
        if op == "fwd":
            shapes_ = dict(A=(M, K), B=(N, K))
            f = lambda a, b: a @ b.t()
        elif op == "dgrad":
            shapes_ = dict(A=(M, N), B=(N, K))
            f = lambda a, b: a @ b
        else:
            shapes_ = dict(A=(M, N), B=(M, K))
            f = lambda a, b: a.t() @ b
        if c["random"]:
            a = torch.randn(shapes_["A"], generator=gen, device=dev, dtype=torch.float32)
            b = torch.randn(shapes_["B"], generator=gen, device=dev, dtype=torch.float32)
            if eng == "bf16":
                a, b = a.to(bf), b.to(bf)
            av, bv = a.double(), b.double()
            if eng == "x3":
                ap = torch.zeros((3,) + tuple(a.shape), dtype=bf, device=dev)
                bp = torch.zeros((3,) + tuple(b.shape), dtype=bf, device=dev)
                C.split_x3(a.contiguous(), ap)
                C.split_x3(b.contiguous(), bp)
                A, B = operand(av, eng, [ap[i].double() for i in range(3)]), operand(bv, eng, [bp[i].double() for i in range(3)])
            else:
                A, B = operand(av, eng), operand(bv, eng)
            ref = f(av, bv)
            denom = f(av.abs(), bv.abs())
        elif eng == "x3":
            ap, bp = x3_planes(shapes_["A"], c["sq"]), x3_planes(shapes_["B"], c["sq"])
            ref = mm6(ap, bp, f)
            A, B = operand(ap[0], eng, ap), operand(bp[0], eng, bp)
            av, bv = ap, bp
        else:
            av, bv = ints(shapes_["A"], r), ints(shapes_["B"], r)
            if hot:
                av[3::8] = ints(av[3::8].shape, 30)
            ref = f(av, bv)
            A, B = operand(av, eng, pad=c["pad"]), operand(bv, eng, pad=c["pad"])
        # spot check of the fp64 device reference: first and last output rows on the CPU
        if not c["random"]:
            sel = (lambda t: t[[0, -1]].cpu()) if op != "wgrad" else (lambda t: t[:, [0, -1]].cpu())
            want_cpu = mm6([sel(x) for x in av], [x.cpu() for x in bv], f) if eng == "x3" else f(sel(av), bv.cpu())
            if not torch.equal(want_cpu, ref[[0, -1]].cpu()):
                return "FAIL the device fp64 reference differs from the CPU in its first or last row"
        rows, cols = ref.shape
        outdt = {"f32": torch.float32, "bf16": bf, "x3": bf}[out]
        obuf, Y = buffer(rows, cols, outdt, CANARY, planes=3 if out == "x3" else 0, pad=c["pad"])
        extra = ""
        if op == "fwd":
            bias = None
            if c["bias"]:
                bv_ = ints((N,), 8)
                bbuf = torch.full((N + 2,), float("nan"), device=dev)
                bbuf[:N] = bv_.float()
                bias = bbuf[:N]
                ref = ref + bv_
            if c["relu"]:
                ref = torch.clamp_min(ref, 0.0)
            C.linear_fwd(A, B, bias, Y, M, N, K, C.ACT_RELU if c["relu"] else C.ACT_NONE, dtype)
        elif op == "dgrad":
            ap_ = None
            if c["mask"]:
                mv = mask_values((M, K))
                ap_ = operand(mv, "f32" if eng == "f32" else "bf16")
                ref = torch.where(mv > 0, ref, torch.zeros_like(ref))
            C.linear_dgrad(A, B, ap_, Y, M, N, K, dtype)
        else:
            dbbuf = None
            if c["db"]:
                dbbuf = torch.full((N + 2,), CANARY, device=dev)
            if c["sq"]:
                slots = C.linear_wgrad_sq_slots(dev, M, N, K, dtype)
                part = torch.full((slots + 2,), CANARY, dtype=torch.float64, device=dev)
                sq = ref * ref
                chunks = torch.nn.functional.pad(sq, (0, (-cols) % 32)).reshape(rows, -1, 32).sum(-1)
                assert float(chunks.max()) < 2 ** 24, "sum-of-squares case whose fp32 partial sums would round"
                C.linear_wgrad_sq(A, B, Y, M, N, K, dtype, part[:slots])
            else:
                C.linear_wgrad(A, B, Y, dbbuf[:N] if dbbuf is not None else None, M, N, K, dtype)
        torch.cuda.synchronize()
        if not check_canary(obuf, rows, cols, out == "x3"):
            return "FAIL output guard rows or padding columns overwritten"
        if c["random"]:
            err = (Y.double() - ref).abs()
            ratio = float((err / denom.clamp_min(1e-300)).max())
            if ratio > RANDOM_BOUND[eng]:
                return "FAIL ratio=%.3e above the bound %.1e" % (ratio, RANDOM_BOUND[eng])
            return "ok ratio=%.3e" % ratio
        if out == "x3":
            h, m, l = (Y[i].double() for i in range(3))
            bad = ((h + m + l) != ref) | (Y[0].float() != ref.float().to(bf).float())
        elif out == "bf16":
            bad = Y.float() != ref.float().to(bf).float()
            n_round = int((ref.float().to(bf).double() != ref).sum())
            if n_round == 0:
                return "FAIL no bf16 rounding exercised"
            extra = " rounded=%d" % n_round
        else:
            bad = Y.double() != ref
        if bool(bad.any()):
            idx = bad.nonzero()
            r0, c0 = int(idx[0, 0]), int(idx[0, 1])
            got = float(Y[0][r0, c0] if out == "x3" else Y[r0, c0])
            return "FAIL %d wrong elements, rows %d..%d, cols %d..%d, first (%d, %d): got %r want %r" % (
                len(idx), int(idx[:, 0].min()), int(idx[:, 0].max()), int(idx[:, 1].min()), int(idx[:, 1].max()), r0, c0, got,
                float(ref[r0, c0]))
        if op == "wgrad" and c["db"]:
            dbw = A.double().sum(0)
            if not torch.equal(dbbuf[:N].double(), dbw) or not bool((dbbuf[N:] == CANARY).all()):
                return "FAIL column sums"
        if op == "wgrad" and c["sq"]:
            if float(part[:slots].sum()) != float((ref * ref).sum()) or not bool((part[slots:] == CANARY).all()):
                return "FAIL sum of squares %r, want %r" % (float(part[:slots].sum()), float((ref * ref).sum()))
        return "ok" + extra

    def prefetch_cases():
        """Weight prefetch (PDL on): a forward after a weight rewrite on the same stream, or on a side stream followed by an
        event wait and codae_weights_written, must read the new weights."""
        M, N, K = 128, 1536, 1536
        X = operand(ints((M, K), 3), "bf16")
        res = {}
        for how in ("cast same stream", "adam same stream", "cast side stream"):
            w_old = ints((N, K), 3)
            w_old[w_old.abs() < 2] = 2.0                       # |w| >= 2: one Adam step of lr 1 keeps it a nonzero integer
            wb = w_old.to(bf).reshape(-1).contiguous()
            W = wb.view(N, K)
            Y1 = torch.full((M, N), CANARY, device=dev)
            Y2 = torch.full((M, N), CANARY, device=dev)
            C.linear_fwd(X, W, None, Y1, M, N, K, C.ACT_NONE, C.BF16)
            main = torch.cuda.current_stream()
            if how.startswith("cast"):
                src = (-w_old).float().reshape(-1).contiguous()
                if how.endswith("side stream"):
                    side = torch.cuda.Stream(device=dev)
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        C.cast_bf16(src, wb)
                        ev = torch.cuda.Event()
                        ev.record(side)
                    main.wait_event(ev)
                    C.weights_written(dev)
                else:
                    C.cast_bf16(src, wb)
            else:
                pf = w_old.float().reshape(-1).contiguous()
                g = torch.sign(pf)
                m, v = torch.zeros_like(pf), torch.zeros_like(pf)
                C.adam_step(pf, g, m, v, wb, 1.0, 0.9, 0.999, 1e-8, 0.0, 1, -1.0, None, 1.0)
            C.linear_fwd(X, W, None, Y2, M, N, K, C.ACT_NONE, C.BF16)
            torch.cuda.synchronize()
            w_new = W.double()
            ok = bool((w_new == torch.round(w_new)).all()) and not bool((w_new == w_old).any())
            ok = ok and torch.equal(Y1.double(), X.double() @ w_old.t()) and torch.equal(Y2.double(), X.double() @ w_new.t())
            res[how] = ok
        return res

    saved = {o: C.get_option(dev, i) for o, i in opt_ids.items()}
    print("SMS %d" % sm, flush=True)
    try:
        for c in case_matrix(sm):
            print("CASE %s" % c["id"], flush=True)
            for o, i in opt_ids.items():
                C.set_option(dev, i, 0 if o in c["run_off"] else 1)
            gen.manual_seed(zlib.crc32(c["id"].encode()))
            try:
                msg = run_case(c)
            except Exception as e:  # a refused call or a broken precondition is a failure of that case
                msg = "FAIL %s: %s" % (type(e).__name__, str(e).replace("\n", " ")[:300])
            for o, i in opt_ids.items():
                C.set_option(dev, i, saved[o])
            print("RESULT %s %s" % (c["id"], msg), flush=True)
        gen.manual_seed(12345)
        for how, ok in prefetch_cases().items():
            print("PREFETCH %s %s" % (how, "ok" if ok else "FAIL"), flush=True)
    finally:
        for o, i in opt_ids.items():
            C.set_option(dev, i, saved[o])
    print("DONE", flush=True)


if __name__ == "__main__":
    if not os.environ.get("CODAE_DEBUG_PLAN"):
        sys.exit("set CODAE_DEBUG_PLAN=1: the library reads it once, and the plan lines are part of the output")
    _run()
