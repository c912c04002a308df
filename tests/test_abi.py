"""CPU: the C-ABI library loads, exports every symbol include/codae_b200.h declares, the ctypes table matches the
header's arity, and the product fails loudly (never falls back) without a GPU."""
import os
import re
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "codae_b200.h")


def header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int|int64_t|size_t|const char\*)\s+(codae_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        n = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
        out[m.group(1)] = n
    return out


def test_header_vs_ctypes_table():
    from codae import _C
    fns = header_functions()
    assert len(fns) >= 25
    assert set(fns) == set(_C.SIGNATURES), set(fns) ^ set(_C.SIGNATURES)
    for name, n in fns.items():
        assert len(_C.SIGNATURES[name][1]) == n, name


def test_option_enum_matches_python_constants():
    """enum codae_option in the header vs the OPT_* constants the Python side passes to codae_ctx_set_option."""
    from codae import _C
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    body = re.search(r"enum\s+codae_option\s*\{(.*?)\}", src, flags=re.S).group(1)
    enum = {m.group(1): int(m.group(2)) for m in re.finditer(r"CODAE_(OPT_\w+)\s*=\s*(\d+)", body)}
    assert len(enum) >= 7 and sorted(enum.values()) == list(range(len(enum)))
    for name, value in enum.items():
        assert getattr(_C, name) == value, name


def test_library_exports_every_symbol():
    from codae import _C
    lib = _C.lib()
    for name in header_functions():
        assert hasattr(lib, name), name
    assert lib.codae_version() == 100
    out = subprocess.run(["nm", "-D", "--defined-only", _C.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (codae_\w+)", out))
    assert set(header_functions()) <= exported


def test_sass_is_blackwell_native():
    """tcgen05.mma / tcgen05.ld / TMA show up as UTCHMMA / LDTM / UTMALDG in the sm_100a SASS."""
    from codae import _C
    # the Makefile calls nvcc by its full path, so the toolkit's bin directory need not be on PATH
    from torch.utils.cpp_extension import CUDA_HOME
    cuobjdump = shutil.which("cuobjdump") or os.path.join(CUDA_HOME or "/usr/local/cuda", "bin", "cuobjdump")
    r = subprocess.run([cuobjdump, "-sass", _C.LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in r.stdout
    for mnem in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnem in r.stdout, mnem


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_gpu_fails_loudly():
    import ctypes
    from codae import _C
    out = ctypes.c_void_p()
    rc = _C.lib().codae_ctx_create(0, ctypes.byref(out))
    assert rc == _C.EARCH and not out.value
    assert b"no CPU path" in _C.lib().codae_last_error(None)
    with pytest.raises(RuntimeError):
        _C.ctx()
    from codae.model import EmbeddingDenoisingAutoencoder
    m = EmbeddingDenoisingAutoencoder(48, 48, 16, 2, 2, False)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(2, 48))
    from codae.tool import Corrupter
    c = Corrupter(4, [dict(size=16, position=16 * i) for i in range(3)], 1, torch.device("cpu"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        c.get_masks((0, 1), 0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mui-deepautoencoder_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                s = open(os.path.join(d, f)).read()
                assert "oracle" not in s.replace("# oracle", ""), os.path.join(d, f)


def test_tiny_layer_struct_layout_matches_header(tmp_path):
    """codae._C.TinyLayer mirrors struct codae_tiny_layer: same size and field offsets as the C compiler sees them."""
    import ctypes
    from codae import _C
    tfields = [f[0] for f in _C.TinyLayer._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "codae_b200.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(codae_tiny_layer));\n' +
                   "".join('  printf(" %%zu", offsetof(codae_tiny_layer, %s));\n' % f.rstrip("_") for f in tfields) +
                   '  printf("\\n");\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    want = [ctypes.sizeof(_C.TinyLayer)] + [getattr(_C.TinyLayer, f).offset for f in tfields]
    assert got == want, (got, want)


def test_dp_peers_struct_layout_matches_header(tmp_path):
    """codae._C.DpPeers mirrors struct codae_dp_peers (the pointer tables of the data-parallel peer kernel)."""
    import ctypes
    from codae import _C
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "codae_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu %d %d\\n", sizeof(codae_dp_peers), offsetof(codae_dp_peers, world), '
                   'offsetof(codae_dp_peers, rank), offsetof(codae_dp_peers, grads), offsetof(codae_dp_peers, w_out), '
                   'offsetof(codae_dp_peers, signals), offsetof(codae_dp_peers, grads_mc), offsetof(codae_dp_peers, w_mc), '
                   'CODAE_DP_MAX_WORLD, CODAE_DP_SIGNAL_BYTES);\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    P = _C.DpPeers
    assert got == [ctypes.sizeof(P), P.world.offset, P.rank.offset, P.grads.offset, P.w_out.offset, P.signals.offset,
                   P.grads_mc.offset, P.w_mc.offset, _C.DP_MAX_WORLD, _C.DP_SIGNAL_BYTES], got


def test_dp_shard_arithmetic():
    """codae_dp_shard_elems: shards are multiples of 8 elements, cover [0, n) and never overlap (host arithmetic, no GPU)."""
    from codae import _C
    for n in (0, 8, 64, 792 // 8 * 8, 23_608_320, 167_813_120, 1_000_000 // 8 * 8):
        for world in (1, 2, 3, 4, 8):
            S = _C.dp_shard_elems(n, world)
            assert S % 8 == 0 and S * world >= n and (world == 1 or S * (world - 1) < n + 8 * world)
            spans = [(min(n, r * S), min(n, (r + 1) * S)) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
