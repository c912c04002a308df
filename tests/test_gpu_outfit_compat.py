"""GPU tests of outfit compatibility scoring (codae_outfit_loo_error; CompatibilityScorer.score_local / score; compatibility_auc;
4_complementarity_inference.py --mode compat).  Every (outfit, slot) row is the outfit with that slot multiplied by 0 (built by
codae_corrupt_fwd) going through the model's GEMM chain; a GEMM row depends only on that row and on the launch's 128-row tile count,
so at a fixed chunk layout an outfit's results do not depend on the other outfits of its chunk."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
ENGINES = ["fp32", "fp32_simt", "bf16"]
RTOL = {"fp32": 1e-5, "fp32_simt": 1e-5, "bf16": 1e-2}


def _model(S, E, dtype, seed, z=96, nin=2, nout=2):
    from codae.model import EmbeddingDenoisingAutoencoder
    torch.manual_seed(seed)
    model = EmbeddingDenoisingAutoencoder(S * E, z, E, nin, nout, False)
    for lin in model.linears():
        torch.nn.init.uniform_(lin.bias, -0.05, 0.05)
    W = [lin.weight.detach().clone() for lin in model.linears()]
    b = [lin.bias.detach().clone() for lin in model.linears()]
    return model.to(DEV).set_compute_dtype(dtype), W, b


def _bits_equal(a, b):
    a, b = a.cpu().contiguous(), b.cpu().contiguous()
    if a.dtype == torch.int64:
        return torch.equal(a, b)
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _oracle_loo(W, b, relu, outfits, E):
    """fp64 restatement: err[i, s] = || DAE(outfit i with slot s * 0)[slot s] - outfit i [slot s] ||^2, [Q, S] float64 (CPU)."""
    dev = outfits.device
    x = outfits.double()
    Q, io = x.shape
    S = io // E
    Wd = [w.to(dev).double() for w in W]
    bd = [v.to(dev).double() for v in b]
    err = torch.empty((Q, S), dtype=torch.float64, device=dev)
    for s in range(S):
        m = torch.ones(io, dtype=torch.float64, device=dev)
        m[s * E:(s + 1) * E] = 0
        h = x * m
        for w, v, r in zip(Wd, bd, relu):
            h = h @ w.T + v
            if r:
                h = torch.relu(h)
        err[:, s] = ((h[:, s * E:(s + 1) * E] - x[:, s * E:(s + 1) * E]) ** 2).sum(1)
    return err.cpu()


def _check_score_odd(err, score, odd):
    """score is the fp32 slot-order sum of the returned err and odd its first argmax, bit for bit (NaN rule: score NaN, odd -1)."""
    err, score, odd = err.cpu(), score.cpu(), odd.cpu()
    want_s = torch.zeros(err.shape[0], dtype=torch.float32)
    for s in range(err.shape[1]):
        want_s = want_s + err[:, s]
    nan = torch.isnan(err).any(1)
    want_s[nan] = float("nan")
    want_o = torch.argmax(torch.where(nan.view(-1, 1), torch.zeros_like(err), err), dim=1)   # torch.argmax: first maximum
    want_o[nan] = -1
    assert _bits_equal(score, want_s)
    assert torch.equal(odd, want_o)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("S,E,Q", [(2, 64, 1), (3, 64, 7), (3, 64, 300), (8, 32, 5000)])
@pytest.mark.parametrize("chunk", [250, 1000, 8192])
def test_matches_fp64_oracle(engine, S, E, Q, chunk):
    from codae.tool.inference import CompatibilityScorer
    model, W, b = _model(S, E, engine, 100 + S)
    g = torch.Generator(device=DEV).manual_seed(Q + S)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    sc = CompatibilityScorer(model, E, chunk=chunk)
    err, score, odd = sc.score_local(outfits)
    ref = _oracle_loo(W, b, model.relu, outfits, E)
    assert err.shape == (Q, S) and score.shape == (Q,) and odd.shape == (Q,)
    np.testing.assert_allclose(err.cpu().double().numpy(), ref.numpy(), rtol=RTOL[engine], atol=1e-6)
    _check_score_odd(err, score, odd)
    # odd agrees with the oracle's argmax wherever the top two errors are apart by more than the tolerance
    top2 = ref.topk(2 if S > 1 else 1, dim=1).values
    clear = (top2[:, 0] - top2[:, -1]) > 4 * RTOL[engine] * top2[:, 0]
    assert torch.equal(odd.cpu()[clear], ref.argmax(1)[clear])


@pytest.mark.parametrize("engine", ENGINES)
def test_results_do_not_depend_on_the_rest_of_the_chunk(engine):
    """chunk = 60 rows = 20 outfits of 3 slots, Q = 40: the other outfits of the target's chunk are replaced, then the chunk is
    permuted (the target moves); its err / score / odd stay bit-identical.  Two runs on the same input are identical."""
    from codae.tool.inference import CompatibilityScorer
    S, E, Q, t = 3, 64, 40, 5
    model, _, _ = _model(S, E, engine, 7)
    sc = CompatibilityScorer(model, E, chunk=60)
    assert sc.chunk_outfits == 20
    g = torch.Generator(device=DEV).manual_seed(8)
    a = torch.rand((Q, S * E), generator=g, device=DEV)
    ra = [x.clone() for x in sc.score_local(a)]
    rb = [x.clone() for x in sc.score_local(a)]
    assert all(_bits_equal(x, y) for x, y in zip(ra, rb))
    b = torch.rand((Q, S * E), generator=g, device=DEV)
    b[t] = a[t]
    rc = [x.clone() for x in sc.score_local(b)]
    assert all(_bits_equal(x[t], y[t]) for x, y in zip(ra, rc))
    perm = torch.randperm(20, generator=torch.Generator().manual_seed(9))
    perm = perm[perm != t]
    perm = torch.cat([perm[:11], torch.tensor([t]), perm[11:]]).to(DEV)    # the target goes to position 11
    c = a.clone()
    c[:20] = a[perm]
    rd = [x.clone() for x in sc.score_local(c)]
    assert all(_bits_equal(x[t], y[11]) for x, y in zip(ra, rd))
    assert all(_bits_equal(x[20:], y[20:]) for x, y in zip(ra, rd))


def _planted_model(S, E, engine):
    """Square layers (z = io), every Linear the identity but the last, which maps every slot to the mean of all slots / (S - 1):
    with slot s hidden (zero) the reconstruction of slot s is the mean of the other slots.  Inputs are >= 0, so the ReLUs pass."""
    from codae.model import EmbeddingDenoisingAutoencoder
    io = S * E
    model = EmbeddingDenoisingAutoencoder(io, io, E, 2, 2, False)
    lins = model.linears()
    with torch.no_grad():
        for lin in lins:
            lin.weight.copy_(torch.eye(io))
            lin.bias.zero_()
        lins[-1].weight.copy_(torch.eye(E).repeat(S, S) / (S - 1))
    return model.to(DEV).set_compute_dtype(engine)


@pytest.mark.parametrize("engine", ENGINES)
def test_planted_odd_item_and_auc(engine):
    from codae import _C
    from codae.tool.inference import CompatibilityScorer, compatibility_auc
    S, E, Q = 5, 32, 200
    model = _planted_model(S, E, engine)
    if engine != "fp32_simt":
        assert model.engine_dtype() == {"fp32": _C.F32X3, "bf16": _C.BF16}[engine]     # widths >= 32: tensor cores
    g = torch.Generator(device=DEV).manual_seed(3)
    v = torch.rand((Q, 1, E), generator=g, device=DEV)
    outfits = v.repeat(1, S, 1)
    j = torch.randint(0, S, (Q,), generator=g, device=DEV)
    outfits[torch.arange(Q, device=DEV), j] += 0.05 + 0.1 * torch.rand((Q, E), generator=g, device=DEV)   # the odd item
    outfits = outfits.view(Q, S * E).contiguous()
    sc = CompatibilityScorer(model, E, chunk=512)
    err, score, odd = (x.clone() for x in sc.score_local(outfits))
    assert torch.equal(odd, j)
    # shuffled copies: slot s of negative q is slot s of outfit perm_s[q]
    neg = outfits.view(Q, S, E).clone()
    for s in range(S):
        p = torch.randperm(Q, generator=torch.Generator().manual_seed(s)).to(DEV)
        neg[:, s] = outfits.view(Q, S, E)[p, s]
    _, neg_score, _ = sc.score_local(neg.view(Q, S * E).contiguous())
    assert compatibility_auc(score, neg_score) == 1.0


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("bad", ["nan", "inf", "-inf"])
def test_non_finite_outfit(engine, bad):
    """A NaN or inf in one slot: that outfit's err is all NaN, its score NaN, its odd -1; the other outfits of its chunk are
    bit-identical to a run without it."""
    from codae.tool.inference import CompatibilityScorer
    S, E, Q = 3, 64, 30
    model, _, _ = _model(S, E, engine, 17)
    sc = CompatibilityScorer(model, E, chunk=300)
    g = torch.Generator(device=DEV).manual_seed(18)
    a = torch.rand((Q, S * E), generator=g, device=DEV)
    ra = [x.clone() for x in sc.score_local(a)]
    b = a.clone()
    b[4, 1 * E + 7] = float(bad)
    err, score, odd = (x.clone() for x in sc.score_local(b))
    assert bool(torch.isnan(err[4]).all()) and bool(torch.isnan(score[4])) and int(odd[4]) == -1
    keep = torch.arange(Q, device=DEV) != 4
    assert _bits_equal(err[keep], ra[0][keep]) and _bits_equal(score[keep], ra[1][keep]) and torch.equal(odd[keep], ra[2][keep])


def test_score_local_does_not_synchronise():
    from codae.tool.inference import CompatibilityScorer
    S, E = 3, 64
    model, _, _ = _model(S, E, "bf16", 5)
    sc = CompatibilityScorer(model, E, chunk=64)
    outfits = torch.rand((50, S * E), device=DEV)
    sc.score_local(outfits)                      # first call allocates
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        sc.score_local(outfits)
        sc.score_local(outfits[:7])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()


def test_bad_inputs_raise():
    from codae.tool.inference import CompatibilityScorer
    S, E = 3, 64
    model, _, _ = _model(S, E, "fp32", 1)
    with pytest.raises(Exception, match="chunk"):
        CompatibilityScorer(model, E, chunk=2)
    sc = CompatibilityScorer(model, E)
    o = torch.rand(4, S * E, device=DEV)
    for bad, match in ((o.double(), "float32"), (o[:, 1:], "shape"), (o[0], "shape"), (o[:0], "shape"), (o.cpu(), "device"),
                       (o.cpu().numpy(), "float32")):
        with pytest.raises(RuntimeError, match=match):
            sc.score_local(bad)


def _guarded(bufs, nbytes, guard=4096):            # 0xff bytes: NaN as float32, -1 as integers
    buf = torch.full((guard + nbytes + guard,), 255, dtype=torch.uint8, device=DEV)
    bufs.append(buf)
    return buf[guard:guard + nbytes]


def test_outputs_stay_in_bounds_and_bad_arguments_are_rejected():
    """err / score / odd inside NaN-filled guarded allocations: exactly the [Q, S] / [Q] entries are written, the guards stay as
    they were; CODAE_EINVAL for NULL pointers, Q < 1, S outside [1, 64], E % 4 != 0, pitches below S E and misaligned buffers."""
    from codae import _C
    from codae.tool.inference import CompatibilityScorer
    S, E, Q, guard = 3, 64, 37, 4096
    io = S * E
    model, _, _ = _model(S, E, "fp32", 71)
    outfits = torch.rand((Q, io), device=DEV)
    ref = [x.clone() for x in CompatibilityScorer(model, E).score_local(outfits)]
    # slot-major reconstructions from the autograd path (predict_slot's forward), errors through the C ABI into guarded outputs
    y = torch.empty((S * Q, io), device=DEV)
    for s in range(S):
        m = torch.ones_like(outfits)
        m[:, s * E:(s + 1) * E] = 0
        with torch.no_grad():
            y[s * Q:(s + 1) * Q] = model(model.corrupt(input_data=outfits, mask=m))
    bufs = []
    err = _guarded(bufs, Q * S * 4).view(torch.float32).view(Q, S)
    score = _guarded(bufs, Q * 4).view(torch.float32)
    odd = _guarded(bufs, Q * 8).view(torch.int64)
    before = [x.clone() for x in bufs]
    _C.outfit_loo_error(outfits, S, E, y, err, score, odd)
    torch.cuda.synchronize()
    for bb, b0 in zip(bufs, before):
        assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])
    assert not bool(torch.isnan(err).any()) and not bool(torch.isnan(score).any()) and bool((odd >= 0).all())
    _check_score_odd(err, score, odd)
    np.testing.assert_allclose(err.cpu().numpy(), ref[0].cpu().numpy(), rtol=1e-5, atol=1e-6)
    c, L, P, st = _C.ctx(DEV), _C.lib(), _C.p, _C.stream()

    def call(**kw):
        a = dict(o=P(outfits), ldo=io, Q=Q, S=S, E=E, y=P(y), ldy=io, err=P(err), score=P(score), odd=P(odd))
        a.update(kw)
        return L.codae_outfit_loo_error(c, a["o"], a["ldo"], a["Q"], a["S"], a["E"], a["y"], a["ldy"], a["err"], a["score"],
                                        a["odd"], st)
    assert call() == _C.OK
    odd_ptr = odd.data_ptr()
    for kw in (dict(o=None), dict(y=None), dict(err=None), dict(score=None), dict(odd=None), dict(Q=0), dict(Q=-1), dict(S=0),
               dict(S=65), dict(E=62), dict(E=0), dict(ldo=io - 1), dict(ldy=io - 4), dict(o=outfits.data_ptr() + 2),
               dict(y=y.data_ptr() + 1), dict(err=err.data_ptr() + 2), dict(odd=odd_ptr + 4)):
        assert call(**kw) == _C.EINVAL, kw
    torch.cuda.synchronize()
    for bb, b0 in zip(bufs, before):
        assert torch.equal(bb[:guard], b0[:guard]) and torch.equal(bb[-guard:], b0[-guard:])


@pytest.mark.parametrize("engine", ["bf16", "fp32"])
def test_embedding_size(engine):
    """embedding.yaml's model (3 slots x 512, 10 x Linear(1536, 1536)) at Q = 10 000, 64 outfits checked against fp64."""
    from codae.tool.inference import CompatibilityScorer
    S, E, Q = 3, 512, 10_000
    model, W, b = _model(S, E, engine, 61, z=1536, nin=4, nout=4)
    assert len(model.dims) == 10
    g = torch.Generator(device=DEV).manual_seed(62)
    outfits = torch.rand((Q, S * E), generator=g, device=DEV)
    err, score, odd = CompatibilityScorer(model, E).score_local(outfits)
    _check_score_odd(err, score, odd)
    pick = torch.randperm(Q, generator=torch.Generator().manual_seed(63))[:64].to(DEV)
    ref = _oracle_loo(W, b, model.relu, outfits[pick], E)
    np.testing.assert_allclose(err[pick].cpu().double().numpy(), ref.numpy(), rtol=RTOL[engine], atol=1e-6)


def _script(tmp_path, *extra):
    args = [os.path.join(PKG, "script", "4_complementarity_inference.py"), "--config", os.path.join(PKG, "config", "embedding.yaml"),
            "--synthetic", "3000", "--queries", "64", "--mode", "compat", "--dtype", "bf16"] + list(extra)
    r = subprocess.run([sys.executable] + args, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_script_compat_mode(tmp_path):
    res = _script(tmp_path)
    assert res["mode"] == "compat" and res["slots"] == 3 and "auc" not in res
    assert len(res["score"]) == 64 and len(res["odd_slot"]) == 64 and all(len(r) == 3 for r in res["slot_errors"])
    assert all(0 <= o < 3 for o in res["odd_slot"])
    for sc, row, o in zip(res["score"], res["slot_errors"], res["odd_slot"]):
        assert abs(sc - sum(row)) <= 1e-5 * abs(sc) and row[o] == max(row)
    neg = _script(tmp_path, "--compat_negatives")
    assert 0.0 <= neg["auc"] <= 1.0
    assert neg["score"] == res["score"] and neg["odd_slot"] == res["odd_slot"]


DIST = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from codae.model import EmbeddingDenoisingAutoencoder
from codae.tool.inference import CompatibilityScorer, shard_rows
dist.init_process_group("nccl")
r, G = dist.get_rank(), dist.get_world_size()
torch.cuda.set_device(r)
dev = torch.device("cuda", r)
S, E, Q = 3, 64, 101
torch.manual_seed(5)
model = EmbeddingDenoisingAutoencoder(S * E, 96, E, 2, 2, False).to(dev).set_compute_dtype("bf16")
outfits = torch.rand((Q, S * E), generator=torch.Generator().manual_seed(6)).to(dev)
sc = CompatibilityScorer(model, E, chunk=60)
err, score, odd = (t.clone() for t in sc.score(outfits))
assert err.shape == (Q, S) and score.shape == (Q,) and odd.shape == (Q,)
for q in range(G):
    lo, n = shard_rows(Q, G, q)
    e, s, o = sc.score_local(outfits[lo:lo + n])
    assert torch.equal(e.view(torch.int32), err[lo:lo + n].view(torch.int32)), q
    assert torch.equal(s.view(torch.int32), score[lo:lo + n].view(torch.int32)) and torch.equal(o, odd[lo:lo + n]), q
# more ranks than outfits: the empty slices still take part in the gather
e1, s1, o1 = (t.clone() for t in sc.score(outfits[:1]))
e0, s0, o0 = sc.score_local(outfits[:1])
assert torch.equal(e1.view(torch.int32), e0.view(torch.int32)) and torch.equal(o1, o0)
dist.barrier()
dist.destroy_process_group()
if r == 0:
    print("COMPAT DIST OK")
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_score_on_two_gpus(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "compat_dist.py"
    script.write_text(DIST)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), PKG]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "COMPAT DIST OK" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
