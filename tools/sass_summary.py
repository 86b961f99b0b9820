"""SASS evidence for the tcgen05 / TMA / TMEM kernels: opcode counts per kernel entry of the built conv_umma.o.

    python tools/sass_summary.py > profiles/r2_sass_summary.txt

UTCHMMA = tcgen05.mma (bf16 -> fp32 in TMEM), UTMALDG = cp.async.bulk.tensor (TMA tile load), LDTM = tcgen05.ld
(TMEM -> registers), UTCBAR = tcgen05.commit (MMA completion -> mbarrier), SYNCS = mbarrier ops, ELECT = elect.sync,
USETMAXREG = setmaxnreg (register re-allocation between warpgroups), LDL / STL = local-memory (spill) traffic.
"""
import re
import subprocess
import sys
from collections import Counter, OrderedDict
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
OPS = ("UTCHMMA", "UTMALDG", "LDTM", "UTCBAR", "SYNCS", "ELECT", "USETMAXREG", "REDG", "ATOMG", "LDG", "STG", "LDS", "STS",
       "LDL", "STL")


def demangle(name: str) -> str:
    try:
        out = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
    except FileNotFoundError:
        return name
    out = re.sub(r"mvlm::\(anonymous namespace\)::", "", out)
    return re.sub(r"\(.*", "", out)


def main():
    obj = "conv_umma.o"
    path = ROOT / "mvlm_b200" / "build" / obj
    sass = subprocess.run(["cuobjdump", "-sass", str(path)], capture_output=True, text=True, check=True).stdout
    funcs = OrderedDict()
    cur = None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(demangle(m.group(1)), Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur is not None:
            cur["total"] += 1
            op = m.group(1)
            for k in OPS:
                if op.startswith(k):
                    cur[k] += 1
    print(f"== mvlm_b200/build/{obj}  (cuobjdump -sass, sm_100a), {len(funcs)} kernel entries")
    print("   " + " ".join(f"{k:>9s}" for k in ("instr",) + OPS) + "  kernel")
    for name, c in funcs.items():
        print("   " + " ".join(f"{c[k]:9d}" for k in ("total",) + OPS) + "  " + name)
    tot = Counter()
    for c in funcs.values():
        tot.update(c)
    print("   " + " ".join(f"{tot[k]:9d}" for k in ("total",) + OPS) + "  (sum)")
    print()


if __name__ == "__main__":
    sys.exit(main())
