#!/usr/bin/env python
"""What the run-time specialised fused Gram kernel executes per sample, counted in the SASS of the cubin NVRTC makes for a chain (no GPU needed):

  python tools/gram_jit_sass_counts.py      -> profiles/gram_jit_sass.json

For C6 and C7 (rosdyn_b200.fixtures), rdb_gram_specialised_cubin compiles gram_fused_kernel<K, SLOTS, true, XC> against the chain's folded
constants for sm_100a, as a Gram call on a B200 does: the rigid-body kernel (XC = 0) and the extended model with a two-column component
(friction) on every joint (XC = 2, tools/bench_ext.py), each also as gram_fused_weighted_kernel (the weighted normal equations: the MMA warps
scale the A operands of every k-step by the weights, counted as mma_dmul_per_4_samples).  The counts are taken as in tools/sass_counts.py (generator = the code in front of the
first DMMA), next to the precompiled kernel's from profiles/gram_fused_sass.json; registers and spills come from cuobjdump -res-usage."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sass_stalls  # noqa: E402
from rosdyn_b200 import _lib, fixtures  # noqa: E402
from rosdyn_b200.descriptor import to_ctypes  # noqa: E402

KPW = 2
CHAINS = {"c6": "gram_fused_kernel<6, 4, true, 0", "c7": "gram_fused_kernel<7, 3, true, 0", "c6_ext": "gram_fused_kernel<6, 4, true, 2",
          "c7_ext": "gram_fused_kernel<7, 3, true, 2", "c6_weighted": "gram_fused_weighted_kernel<6, 4, true, 0",
          "c7_weighted": "gram_fused_weighted_kernel<7, 3, true, 0", "c6_ext_weighted": "gram_fused_weighted_kernel<6, 3, true, 2",
          "c7_ext_weighted": "gram_fused_weighted_kernel<7, 3, true, 2"}


def count(cubin: str):
    sass = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout.splitlines()
    ins = sass_stalls.parse(sass)
    first_dmma = next((k for k, i in enumerate(ins) if "DMMA" in i["text"]), len(ins))
    gen = ins[:first_dmma]
    cnt = {op: sum(1 for i in gen if re.match(r"(@!?U?P\d+\s+)?" + op + r"\b", i["text"])) for op in ("DFMA", "DMUL", "DADD")}
    dmma = sum(1 for i in ins if "DMMA" in i["text"])
    mma_dfma = sum(1 for i in ins[first_dmma:] if re.match(r"(@!?U?P\d+\s+)?DFMA\b", i["text"]))
    mma_dmul = sum(1 for i in ins[first_dmma:] if re.match(r"(@!?U?P\d+\s+)?DMUL\b", i["text"]))
    res = subprocess.run(["cuobjdump", "-res-usage", cubin], capture_output=True, text=True, check=True).stdout
    m = re.search(r"REG:(\d+) STACK:(\d+)", res)
    return {"gen_dp_instr_per_sample": sum(cnt.values()), "gen_flop_per_sample": float(2 * cnt["DFMA"] + cnt["DMUL"] + cnt["DADD"]),
            "gen_ops": cnt, "dmma_total": dmma, "dmma_per_4_samples": dmma / KPW, "mma_dfma_per_4_samples": mma_dfma / KPW,
            "mma_dmul_per_4_samples": mma_dmul / KPW,
            "registers": int(m.group(1)) if m else None, "stack_bytes": int(m.group(2)) if m else None}


def main():
    lib = _lib.load()
    pre = json.load(open(os.path.join(ROOT, "profiles", "gram_fused_sass.json")))
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, kargs in CHAINS.items():
            cdesc, keep = to_ctypes(fixtures.by_name(name.split("_")[0]))
            path = os.path.join(tmp, name + ".cubin")
            why = ctypes.create_string_buffer(4096)
            t0 = time.perf_counter()
            st = lib.rdb_gram_specialised_cubin(ctypes.byref(cdesc), kargs.encode(), b"sm_100a", path.encode(), why, len(why))
            dt = time.perf_counter() - t0
            del keep
            if st != 0:
                raise SystemExit(f"{name}: {lib.rdb_last_error().decode()}")
            r = count(path)
            K, XC = (int(a) for a in kargs.split("<")[1].split(", ")[::3])
            weighted = "weighted" in kargs
            r.update({"kernel": kargs + ", GramJitModel>", "nvrtc_compile_s_cpu": round(dt, 2),
                      # profiles/gram_fused_sass.json counts the rigid-body kernels only
                      "precompiled_gen_dp_instr_per_sample": pre.get(f"K{K}_rev", {}).get("gen_dp_instr_per_sample") if XC == 0 and not weighted else None})
            out[name] = r
            print(f"{name}: generator FP64 instr / sample {r['gen_dp_instr_per_sample']} (precompiled {r['precompiled_gen_dp_instr_per_sample']}; "
                  f"DFMA {r['gen_ops']['DFMA']}, DMUL {r['gen_ops']['DMUL']}, DADD {r['gen_ops']['DADD']}), DMMA per 4 samples "
                  f"{r['dmma_per_4_samples']:.0f}, MMA-side DMUL per 4 samples {r['mma_dmul_per_4_samples']:.1f}, {r['registers']} registers, stack {r['stack_bytes']} B, NVRTC {dt:.1f} s on the host CPU")
    json.dump(out, open(os.path.join(ROOT, "profiles", "gram_jit_sass.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
