#!/usr/bin/env python
"""Forward dynamics on the GPU: the fused entry against the composition a user would otherwise write, in one run.

  python tools/bench_fd.py [--samples 1e8] [--seconds 1.0] [--rounds 3] [--out profiles/fd_bench.json] [--fd-only] [--lib path]

Per chain (C6, C7): device-resident q, Dq, DDq from rdb_fill_uniform (1e8 samples, far beyond L2), tau = rdb_torque_batch(q, Dq, DDq), then
  * fused : rdb_forward_dynamics_batch over all samples, repeated for >= --seconds (CUDA events);
  * comp  : rdb_inertia_batch + rdb_torque_batch(DDq = NULL) + torch.linalg.cholesky / cholesky_solve over [chunk, n, n], chunk by chunk
            (4 M samples) for >= --seconds;
alternating, --rounds times; the median rates and their ratio are reported.  Both outputs are checked against each other and against DDq
(maxabs(x - ref) <= 1e-10 max(maxabs(ref), 1)).  The GPU name, power limit and the SM clock sampled during the timed regions are part of
the result, and the rate is set against the FP64-issue ceiling from the SASS count (tools/fd_sass_counts.py).  --fd-only times the fused
entry alone (A/B between library builds with --lib)."""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from rosdyn_b200 import _lib, fixtures  # noqa: E402

CHUNK = 1 << 22


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
    ap.add_argument("--samples", type=float, default=1e8)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--fd-only", action="store_true")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--chains", default="c6,c7")
    a = ap.parse_args()
    if a.lib:
        _lib.set_library_path(os.path.abspath(a.lib))
    import torch
    from bench import ClockSampler
    from rosdyn_b200.chain import Chain
    assert torch.cuda.is_available(), "tools/bench_fd.py measures on a CUDA device"
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    S = int(a.samples)
    try:
        from fd_sass_counts import count
        sass = {6: count(os.path.join(ROOT, "build", "kernels.o"), 6), 7: count(os.path.join(ROOT, "build", "kernels.o"), 7)}
    except Exception as e:  # noqa: BLE001
        sass = {"error": str(e)}
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "samples": S, "lib": a.lib or "default", "chains": {}}

    def timed(fn, seconds):
        """fn() once per repetition; repetitions for >= seconds; returns (seconds per repetition, clock summary)."""
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
        n = d.n_inputs
        q, dq, ddq = (torch.empty((n, S), dtype=torch.float64, device="cuda") for _ in range(3))
        for k, x in enumerate((q, dq, ddq)):
            _lib.check(lib.rdb_fill_uniform(x.data_ptr(), n, S, S, 0x5EED0000 + 51, k, st))
        tau = torch.empty_like(q)
        s_all = _lib.CSamples(S, S, q.data_ptr(), dq.data_ptr(), ddq.data_ptr(), None)
        _lib.check(lib.rdb_torque_batch(ch._h, ctypes.byref(s_all), tau.data_ptr(), S, st))
        out = torch.empty_like(q)
        info = torch.empty((S,), dtype=torch.int32, device="cuda")
        s_fd = _lib.CSamples(S, S, q.data_ptr(), dq.data_ptr(), None, None)

        def fused():
            _lib.check(lib.rdb_forward_dynamics_batch(ch._h, ctypes.byref(s_fd), tau.data_ptr(), out.data_ptr(), S, info.data_ptr(), st))

        M = torch.empty((n * n, CHUNK), dtype=torch.float64, device="cuda")
        h = torch.empty((n, CHUNK), dtype=torch.float64, device="cuda")
        comp_out = torch.empty((n, CHUNK), dtype=torch.float64, device="cuda")
        n_chunks = S // CHUNK
        state = {"k": 0}

        def comp_chunk(k):
            off = k * CHUNK
            s = _lib.CSamples(CHUNK, S, q.data_ptr() + 8 * off, dq.data_ptr() + 8 * off, None, None)
            _lib.check(lib.rdb_inertia_batch(ch._h, ctypes.byref(s), M.data_ptr(), CHUNK, st))
            _lib.check(lib.rdb_torque_batch(ch._h, ctypes.byref(s), h.data_ptr(), CHUNK, st))
            A = M.view(n, n, CHUNK).permute(2, 1, 0)                     # plane col * n + row -> [sample, row, col]
            L = torch.linalg.cholesky(A)
            b = (tau[:, off:off + CHUNK] - h).T.unsqueeze(-1)
            comp_out.copy_(torch.cholesky_solve(b, L)[..., 0].T)

        def comp():
            comp_chunk(state["k"] % n_chunks)
            state["k"] += 1

        # agreement on the first chunk, and the round trip over all samples
        fused()
        comp_chunk(0)
        torch.cuda.synchronize()
        def rel(x, ref):
            return float((x - ref).abs().max() / max(float(ref.abs().max()), 1.0))
        agree = rel(comp_out, out[:, :CHUNK])
        round_trip = rel(out, ddq)
        bad = int((info != 0).sum())
        rounds = []
        for _ in range(a.rounds):
            t_f, clk_f = timed(fused, a.seconds)
            r = {"fused_G_per_s": S / t_f / 1e9, "fused_clock": clk_f}
            if not a.fd_only:
                t_c, clk_c = timed(comp, a.seconds)
                r.update({"comp_G_per_s": CHUNK / t_c / 1e9, "comp_clock": clk_c})
            rounds.append(r)
            print(name, json.dumps(r), flush=True)
        fr = statistics.median(r["fused_G_per_s"] for r in rounds)
        mhz = statistics.median(r["fused_clock"]["sm_mhz"] or 0.0 for r in rounds)
        c = {"n_inputs": n, "fused_G_samples_per_s": fr, "sm_mhz_fused": mhz, "rounds": rounds, "info_nonzero": bad,
             "max_rel_err_fused_vs_DDq": round_trip, "max_rel_err_fused_vs_comp_chunk0": agree, "agree_1e-10": agree <= 1e-10 and round_trip <= 1e-10}
        if not a.fd_only:
            cr = statistics.median(r["comp_G_per_s"] for r in rounds)
            c.update({"comp_G_samples_per_s": cr, "speedup_fused_over_comp": fr / cr})
        nj = len([j for j in d.joints if j.input_index >= 0])
        if isinstance(sass, dict) and nj in sass and mhz:
            dp = sass[nj]["dp_instr_per_sample"]
            ceil = 148 * 4 * (mhz * 1e6) / 2 * 32 / dp / 1e9   # one DP warp instruction per 2 cycles per SM sub-partition, 32 samples each
            c.update({"dp_instr_per_sample": dp, "fp64_issue_ceiling_G_per_s": ceil, "fraction_of_fp64_ceiling": fr / ceil})
        res["chains"][name] = c
        print(name, json.dumps({k: v for k, v in c.items() if k != "rounds"}), flush=True)
        del q, dq, ddq, tau, out, info, M, h, comp_out
        torch.cuda.empty_cache()
    res["ptxas_sass"] = sass
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "chains"}))


if __name__ == "__main__":
    t0 = time.time()
    main()
    print(f"wall {time.time() - t0:.1f} s")
