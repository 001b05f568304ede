#!/usr/bin/env python3
"""Do two builds of libhw1f.so schedule their time loops the same way?  For every simulation kernel the opcode sequence
from the first to the last Box-Muller MUFU.LG2 (the time loops and what lies between them) is compared between the two libraries: "loops identical"
means a source change stayed in the prologue and the measured difference is not ptxas' instruction order (which is worth
+-2 % on these kernels, DESIGN.md section 4).  Needs only cuobjdump (no GPU).

    python tools/sass_loop_diff.py old.so new.so"""
import difflib
import re
import subprocess
import sys

KERNELS = ("fast_kernel", "bond_curve_kernel", "zbc_kernel", "fused_kernel", "pathwise_kernel", "zbc_sum_kernel",
           "swaption_kernel", "book_vega_kernel")


def functions(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and cur:
            funcs[cur].append(re.sub(r"^@!?U?P\d+\s+", "", m.group(2).strip()).split()[0])
    return funcs


def main(old, new):
    a, b = functions(old), functions(new)
    for name in sorted(a):
        if not any(k in name for k in KERNELS) or name not in b:
            continue
        ia = [i for i, op in enumerate(a[name]) if op.startswith("MUFU.LG2")]
        ib = [i for i, op in enumerate(b[name]) if op.startswith("MUFU.LG2")]
        if not ia or not ib:
            continue
        ta, tb = a[name][ia[0]:ia[-1] + 1], b[name][ib[0]:ib[-1] + 1]
        verdict = "loops identical" if ta == tb else \
            "loops differ (similarity %.3f)" % difflib.SequenceMatcher(None, ta, tb, autojunk=False).ratio()
        short = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.split("(")[0].strip()
        print(f"{short[:64]:64s} instructions {len(a[name]):5d} -> {len(b[name]):5d}   {verdict}")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
