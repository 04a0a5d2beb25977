#!/usr/bin/env python
"""Segmented normal equations on the device: rdb_regressor_gram_segmented_batch against the two ways to get the same systems without it.

    python tools/bench_gram_segmented.py [--samples 16777216] [--seconds 1.0] [--rounds 3] [--out file.json]

For C6 and C7, 2^24 samples in total (3 x 2^24 x n doubles of inputs, far more than the 126 MB L2), cut into segments of 1 024, 4 096,
65 536 and 2^24 samples, the same call alternates, round by round:
  (a) one rdb_regressor_gram_segmented_batch call over all segments;
  (b) one rdb_regressor_gram_batch call per segment (pointer-offset inputs), through ctypes;
  (c) one rdb_regressor_gram_batch call over all samples (one system: the rate the segmented entry approaches).
Rates are samples per second of the median round.  (a) and (b) are compared segment by segment (max |a - b| over max(max |b|, 1)).
A sweep of the work-item length and the wave size (RDB_GRAM_SEG_ITEM_GROUPS, RDB_GRAM_SEG_WAVE_PER_SM) times (a) alone; it is what chose
the defaults of csrc/gram_fused.cu.  The GPU name, its power limit and the SM clock sampled during the timed regions go with the numbers."""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rosdyn_b200 import _lib, fixtures  # noqa: E402

LENGTHS = [1024, 4096, 65536, 1 << 24]
SWEEP = [(64, 4), (64, 8), (128, 4), (128, 8), (256, 8), (128, 16)]  # (groups per item, items per SM per wave)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True,
                             timeout=20).stdout.strip().split(", ")
        return {"name": out[0], "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1 << 24)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chains", default="c6,c7")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from bench import ClockSampler
    from rosdyn_b200.chain import Chain
    assert torch.cuda.is_available(), "tools/bench_gram_segmented.py measures on a CUDA device"
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    S = a.samples
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "sms": sm, "samples": S,
           "inputs": "device-resident, 3 planes x n_inputs x 2^24 doubles (> L2)", "chains": {}}

    def timed(fn, seconds):
        """fn() once per repetition; repetitions for >= seconds; returns (seconds per repetition, clock summary)"""
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        reps = max(1, math.ceil(seconds / (e0.elapsed_time(e1) / 1e3)))
        with ClockSampler(0) as clk:
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps, clk.summary()

    for name in a.chains.split(","):
        d = fixtures.by_name(name)
        ch = Chain(d)
        n, P = d.n_inputs, 10 * d.n_joints
        x = torch.empty((3, n, S), dtype=torch.float64, device="cuda")
        for k in range(3):
            _lib.check(lib.rdb_fill_uniform(x[k].data_ptr(), n, S, S, 0x5EED0000 + 77, k, st))
        s_all = _lib.CSamples(S, S, x[0].data_ptr(), x[1].data_ptr(), x[2].data_ptr(), None)
        G1 = torch.empty((P * P + P + 1,), dtype=torch.float64, device="cuda")
        rows = {}
        for L in LENGTHS:
            K = S // L
            offs = (ctypes.c_int64 * (K + 1))(*range(0, K * L + 1, L))
            Ga = torch.empty((K * (P * P + P + 1),), dtype=torch.float64, device="cuda")
            Gb = torch.empty_like(Ga)
            pa = [ctypes.c_void_p(Ga.data_ptr() + 8 * o) for o in (0, K * P * P, K * P * P + K * P)]
            segs = [_lib.CSamples(L, S, x[0].data_ptr() + 8 * k * L, x[1].data_ptr() + 8 * k * L, x[2].data_ptr() + 8 * k * L, None)
                    for k in range(K)]
            outs = [tuple(ctypes.c_void_p(Gb.data_ptr() + 8 * o) for o in (k * P * P, K * P * P + k * P, K * P * P + K * P + k))
                    for k in range(K)]

            def seg():
                _lib.check(lib.rdb_regressor_gram_segmented_batch(ch._h, ctypes.byref(s_all), None, K, offs, *pa, 0, st))

            def loop():
                for s, o in zip(segs, outs):
                    _lib.check(lib.rdb_regressor_gram_batch(ch._h, ctypes.byref(s), None, *o, 0, st))

            def whole():
                _lib.check(lib.rdb_regressor_gram_batch(ch._h, ctypes.byref(s_all), None, ctypes.c_void_p(G1.data_ptr()),
                                                        ctypes.c_void_p(G1.data_ptr() + 8 * P * P), ctypes.c_void_p(G1.data_ptr() + 8 * (P * P + P)),
                                                        0, st))

            seg()
            loop()
            torch.cuda.synchronize()
            err = float((Ga - Gb).abs().max() / max(float(Gb.abs().max()), 1.0))
            rounds = {"segmented": [], "loop": [], "unsegmented": []}
            clocks = []
            for _ in range(a.rounds):
                for k, fn in (("segmented", seg), ("loop", loop), ("unsegmented", whole)):
                    t, clk = timed(fn, a.seconds)
                    rounds[k].append(S / t / 1e9)
                    clocks.append(clk)
            med = {k: statistics.median(v) for k, v in rounds.items()}
            rows[L] = {"segments": K, "G_samples_per_s": med, "rounds": rounds, "seg_vs_loop": med["segmented"] / med["loop"],
                       "seg_vs_unsegmented": med["segmented"] / med["unsegmented"], "max_rel_diff_seg_vs_loop": err,
                       "kernel_info": None, "sm_mhz_median": statistics.median(c.get("sm_mhz") or 0.0 for c in clocks), "throttle_reasons": sorted({r for c in clocks for r in c.get("reasons", [])})}
            seg()
            flag = ctypes.c_int32(-1)
            buf = ctypes.create_string_buffer(512)
            lib.rdb_chain_gram_kernel_info(ch._h, ctypes.byref(flag), buf, len(buf))
            rows[L]["kernel_info"] = [flag.value, buf.value.decode()[:120]]
            print(f"{name} L={L:>8d} K={K:>6d}: segmented {med['segmented']:.4f}  loop {med['loop']:.4f}  unsegmented {med['unsegmented']:.4f} "
                  f"G samples/s  (seg/loop {rows[L]['seg_vs_loop']:.1f}x, seg/unseg {rows[L]['seg_vs_unsegmented']:.3f}, diff {err:.1e}, "
                  f"{rows[L]['sm_mhz_median']:.0f} MHz)", flush=True)
            # the item length / wave size sweep, segmented entry alone
            sweep = {}
            for ig, wps in SWEEP:
                os.environ["RDB_GRAM_SEG_ITEM_GROUPS"], os.environ["RDB_GRAM_SEG_WAVE_PER_SM"] = str(ig), str(wps)
                t, _ = timed(seg, a.seconds / 2)
                sweep[f"{ig}x32 samples, {wps}/SM"] = S / t / 1e9
            del os.environ["RDB_GRAM_SEG_ITEM_GROUPS"], os.environ["RDB_GRAM_SEG_WAVE_PER_SM"]
            rows[L]["sweep_G_samples_per_s"] = sweep
            print(f"    sweep: " + ", ".join(f"{k}: {v:.4f}" for k, v in sweep.items()), flush=True)
            del Ga, Gb, segs, outs
        res["chains"][name] = rows
        del x
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
