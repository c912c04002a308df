#!/usr/bin/env python
"""SASS mnemonic counts per tensor-core kernel of libcodae_b200.so (cuobjdump -sass, no GPU needed):
    python tools/sass_summary.py > profiles/r02_sass_summary.txt
UTCHMMA = tcgen05.mma (kind::f16), LDTM = tcgen05.ld, UTMALDG / UTMASTG = TMA bulk tensor load / store, UTCBAR = tcgen05.commit,
SYNCS = mbarrier operations, UCGABAR = cluster barrier arrive / wait.

    python tools/sass_summary.py --compare OLD.o NEW.o PATTERN
prints one JSON line per kernel whose name contains PATTERN: its opcode sequence (operands stripped) in two builds of an object
file and whether the sequences are equal -- the check that a refactor left a kernel's instructions as they were."""
import collections
import json
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def functions(path):
    """{demangled kernel name: SASS text} of a cubin-carrying object or library."""
    txt = subprocess.run([CUOBJDUMP, "-sass", path], capture_output=True, text=True).stdout
    out = {}
    for p in re.split(r"\n\s*Function : ", txt)[1:]:
        name = p.split("\n", 1)[0].strip()
        dem = subprocess.run(["c++filt", "-p", name], capture_output=True, text=True).stdout.strip()
        out[dem.replace("(anonymous namespace)::", "")] = p
    return out


def opcodes(sass):
    return re.findall(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", sass)


if len(sys.argv) == 5 and sys.argv[1] == "--compare":
    old, new = functions(sys.argv[2]), functions(sys.argv[3])
    for name in sorted(old):
        if sys.argv[4] in name:
            a, b = opcodes(old[name]), opcodes(new.get(name, ""))
            print(json.dumps({"kernel": name, "old_instructions": len(a), "new_instructions": len(b), "same_opcode_sequence": a == b}))
    raise SystemExit(0)

so = os.path.join(ROOT, "mui-deepautoencoder_b200", "codae", "_lib", "libcodae_b200.so")
print(__doc__.strip().split("\n\n")[0].replace("\n", "\n# ").join(["# ", ""]))
print("%-70s %8s %6s %8s %8s %7s %6s %8s" % ("kernel", "UTCHMMA", "LDTM", "UTMALDG", "UTMASTG", "UTCBAR", "SYNCS", "UCGABAR"))
for dem, p in functions(so).items():
    c = collections.Counter(re.findall(r"\b(UTCHMMA|LDTM|UTMALDG|UTMASTG|UTCBAR|SYNCS|UCGABAR_ARV|UCGABAR_WAIT)\b", p))
    if c["UTCHMMA"] or c["UTMALDG"] or c["LDTM"]:
        print("%-70s %8d %6d %8d %8d %7d %6d %8d" % (dem[:70], c["UTCHMMA"], c["LDTM"], c["UTMALDG"], c["UTMASTG"], c["UTCBAR"],
                                                     c["SYNCS"], c["UCGABAR_ARV"] + c["UCGABAR_WAIT"]))
