"""The GEMM conformance case matrix (tests/_gemm_conformance_cases.py) reaches every required plan cell, according to the
pure-Python mirror of the plan choice, on a 148-SM B200 and on a part with fewer SMs.  No GPU needed: on the B200,
tests/test_gpu_gemm_conformance.py checks the mirror itself against the plans the library logs."""
import pytest

import _gemm_conformance_cases as G


@pytest.mark.parametrize("sm", [148, 132])
def test_case_matrix_covers_every_required_plan_cell(sm):
    cov = G.coverage(sm)
    missing = sorted(G.required_cells() - set(cov))
    assert not missing, missing


def test_mirror_matches_known_plans():
    """The mirror against plans worked out by hand from csrc/gemm_tcgen05.cu and csrc/gemm_simt.cu at 148 SMs."""
    def plan(eng, op, M, N, K, out="f32", **kw):
        return G.expected_plan(148, G.make_case(eng, op, M, N, K, out, **kw))
    # small-batch dgrad of a 1536-wide layer: one-row-tile rule, 12 clusters of 8
    p = plan("bf16", "dgrad", 128, 1536, 1536, mask=True)
    assert (p["bn"], p["gx"], p["gy"], p["nsplit"], p["staged"]) == (128, 12, 1, 8, 1)
    # forward at M = 8192, N = 384: BN = 128, single pass
    p = plan("bf16", "fwd", 8192, 384, 72, "bf16", bias=True, relu=True)
    assert (p["bn"], p["nsplit"], p["staged"], p["persistent"]) == (128, 1, 0, 0)
    # polyvore-shaped layer: CTA pairs on 256 x 256 tiles
    p = plan("bf16", "fwd", 8192, 4096, 4097, "bf16", relu=True)
    assert p == dict(kind="tc", bn=256, persistent=1, pair=1, tma_store=1)
    # augmented weight gradient of a 4096-wide layer at B = 256: 32 x 17 tiles of 128 x 256, more than 2 per SM
    p = plan("bf16", "wgrad", 256, 4096, 4097)
    assert p == dict(kind="tc", bn=256, persistent=1, pair=1, tma_store=1)
    # B = 64, 1536-wide layer: 84 tiles of 128 x 256 < 148 <= 156 tiles of 128 x 128, staged with the bulk store
    p = plan("bf16", "wgrad", 64, 1536, 1537)
    assert (p["bn"], p["nsplit"], p["staged"], p["tma_store"], p["persistent"]) == (128, 1, 1, 1, 0)
    p = plan("x3", "fwd", 100, 200, 4600, relu=True)
    assert (p["nsplit"], p["chunked"]) == (8, 1)
    assert plan("f32", "fwd", 128, 1536, 1536, bias=True)["split"] == 3          # 48 tiles of 64 x 64: 148 // 48 = 3


def test_plan_lines_parse():
    dims, p = G.parse_plan("codae plan: M=128 N=1536 K=1536 BN=128 NP=1 grid 12 x 1 x 8 stages 3 smem 394496 tmem 128 staged 1 "
                           "tma_store 0 chunked 0 occupancy 1")
    assert dims == (128, 1536, 1536) and (p["bn"], p["gx"], p["nsplit"], p["staged"], p["tma_store"]) == (128, 12, 8, 1, 0)
    dims, p = G.parse_plan("codae plan: M=4196 N=2507 K=72 BN=256 persistent pair 1 tma_store 0 ctas 148")
    assert dims == (4196, 2507, 72) and p == dict(kind="tc", bn=256, persistent=1, pair=1, tma_store=0)
    dims, p = G.parse_plan("codae plan: simt M=100 N=200 K=1000 EPI=1 tile 64 split 7")
    assert dims == (100, 200, 1000) and p == dict(kind="simt", tile=64, split=7)
    assert G.parse_plan("RESULT x ok") is None
