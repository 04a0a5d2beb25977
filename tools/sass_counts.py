#!/usr/bin/env python
"""What the fused Gram kernel executes per sample, counted in the SASS of the object that ships (no GPU needed):

  python tools/sass_counts.py            -> profiles/gram_fused_sass.json  (+ profiles/r02_gram_fused_sass_summary.txt)

For every rigid-body instantiation gram_fused_kernel<K, SLOTS, REV, XC = 0>:
  * gen_dp_instr_per_sample : FP64 instructions (DFMA / DMUL / DADD) one generator LANE executes for its sample (a warp instruction serves 32
    samples).  The generator's code is the straight-line region in front of the first DMMA of the kernel (the MMA roles follow it); the
    rarely taken library sincos for |q| > 1e5 is a CALL outside it.
  * gen_flop_per_sample     : DFMA = 2 flop, DMUL / DADD = 1 flop.
  * dmma_per_4_samples      : DMMA.8x8x4 of the MMA roles for one k-step (4 samples) of every joint row = all DMMAs of the kernel / k-steps per
    warp and joint row (GramGeom::KPW = 2: the two tile-parity roles each unroll KPW k-steps of every row).
  * mma_dfma_per_4_samples  : DFMA of the MMA roles (behind the first DMMA) for the same 4 samples: Phi^T tau and tau^T tau accumulated beside
    the tiles (GramGeom TC == 0).
bench.py reads the JSON for roofline.executed."""
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sass_stalls  # noqa: E402

KPW = 2
GENS = 4  # generator warps of every instantiation (GF_GENS)


def main():
    obj = os.path.join(ROOT, "build", "gram_fused.o")
    names = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    funcs = sorted(set(re.findall(r"Function : (\S*gram_fused_kernel\S*)", names)))
    out, lines = {}, []
    for f in funcs:
        dem = subprocess.run(["c++filt", f], capture_output=True, text=True).stdout.strip()
        m = re.search(r"gram_fused_kernel<(\d+), (\d+), (true|false|\(bool\)[01]), (\d+)(?:, rdb::RtModel)?>", dem)
        if not m:
            continue
        K, slots, rev, XC = int(m.group(1)), int(m.group(2)), m.group(3) in ("true", "(bool)1"), int(m.group(4))
        if XC != 0:
            continue
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", f, obj], capture_output=True, text=True).stdout.splitlines()
        ins = sass_stalls.parse(sass)
        first_dmma = next((k for k, i in enumerate(ins) if "DMMA" in i["text"]), len(ins))
        gen = ins[:first_dmma]
        cnt = {op: sum(1 for i in gen if re.match(r"(@!?U?P\d+\s+)?" + op + r"\b", i["text"])) for op in ("DFMA", "DMUL", "DADD")}
        dmma = sum(1 for i in ins if "DMMA" in i["text"])
        mma_dfma = sum(1 for i in ins[first_dmma:] if re.match(r"(@!?U?P\d+\s+)?DFMA\b", i["text"]))
        dp = sum(cnt.values())
        key = f"K{K}_{'rev' if rev else 'gen'}"
        out[key] = {"kernel": dem.split("(")[0].replace("void rdb::", "").replace(", rdb::RtModel>", ">"), "slots": slots, "generator_warps": GENS,
                    "gen_dp_instr_per_sample": dp,
                    # flop per sample: every lane of a generator warp instruction works on its own sample
                    "gen_flop_per_sample": float(2 * cnt["DFMA"] + cnt["DMUL"] + cnt["DADD"]),
                    "gen_ops": cnt, "dmma_total": dmma, "dmma_per_4_samples": dmma / KPW,
                    "mma_dfma_per_4_samples": mma_dfma / KPW}
        lines.append(f"{out[key]['kernel']:48s} generator FP64 instr / sample {dp:5d} (DFMA {cnt['DFMA']}, DMUL {cnt['DMUL']}, DADD {cnt['DADD']}) = "
                     f"{out[key]['gen_flop_per_sample']:.0f} flop;  DMMA.8x8x4 in the kernel {dmma} = {dmma / KPW:.0f} per 4 samples "
                     f"({dmma / KPW * 128:.0f} flop / sample)")
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "profiles", "gram_fused_sass.json"), "w"), indent=1, sort_keys=True)
    open(os.path.join(ROOT, "profiles", "r02_gram_fused_sass_summary.txt"), "w").write(
        "# FP64 work of gram_fused_kernel counted in the SASS of build/gram_fused.o (tools/sass_counts.py); one lane = one sample in the generator\n"
        + "\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
