#!/usr/bin/env python
"""FP64 instructions the forward-dynamics walker executes per sample, counted in the SASS of build/kernels.o (no GPU needed):

  python tools/fd_sass_counts.py [build/kernels.o]

For dyn_kernel<NJ, DYN_FD, REV> (NJ = 6, 7, REV = true: C6 / C7 on the folded chain) it counts DFMA + DMUL + DADD + DSETP (DESIGN.md 3.2's
method) on the path every sample takes: the kernel body up to its final EXIT, without the per-angle trig fallback that the branch
`@P0 BRA P2, <target>` after the vectorised sin/cos skips, and without the subroutines behind the body (the library sincos for |q| > 1e5).
One lane executes these for its own sample; a warp instruction serves 32 samples.  Prints one JSON object."""
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DP = ("DFMA", "DMUL", "DADD", "DSETP")
INS = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9]+)[.\w]*\s*([^;]*);")


def count(obj, nj):
    fn = f"_ZN3rdb10dyn_kernelILi{nj}ELi8ELb1ELb0EEEvNS_8ChainDevIXT_EEENS_10SamplesDevENS_9DynOutDevE"
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", fn, obj], capture_output=True, text=True, check=True).stdout
    ins = [(int(m.group(1), 16), m.group(2) or "", m.group(3), m.group(4)) for m in INS.finditer(sass)]
    end = next(a for a, p, op, _ in ins if op == "EXIT" and not p and a > 0x100)
    skip = None
    for a, p, op, arg in ins:
        m = re.match(r"P\d+, 0x([0-9a-f]+)", arg.strip())
        if op == "BRA" and p.strip() == "@P0" and m:
            skip = (a + 16, int(m.group(1), 16))
            break
    total = sum(1 for a, _, op, _ in ins if op in DP)
    path = sum(1 for a, _, op, _ in ins if op in DP and a <= end and not (skip and skip[0] <= a < skip[1]))
    return {"dp_instr_in_function": total, "dp_instr_per_sample": path, "trig_fallback_skipped": [hex(x) for x in skip] if skip else None}


def main():
    obj = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "build", "kernels.o")
    print(json.dumps({f"dyn_kernel<{nj},DYN_FD,REV>": count(obj, nj) for nj in (6, 7)}, indent=1))


if __name__ == "__main__":
    main()
