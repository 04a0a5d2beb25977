#!/usr/bin/env python
"""Weighted normal equations on the device: rdb_regressor_gram_weighted_batch / rdb_regressor_gram_ext_weighted_batch against the
unweighted entries and against the composition that was the only way to get them before.

    python tools/bench_gram_weighted.py [--samples 16777216] [--seconds 1.0] [--rounds 3] [--out file.json]

For C6 and C7, rigid-body and with a first-order friction component on every joint (the extended model), over 2^24 device-resident samples
(3 x 2^24 x n doubles of inputs plus 2^24 x n of measured torques and of weight planes, far more than the 126 MB L2), the same calls
alternate, round by round, each timed over at least --seconds:
  unweighted   rdb_regressor_gram_batch / rdb_regressor_gram_ext_batch;
  joint        one weight per joint (strides 1, 0);
  sample       one weight per sample (strides 0, 1);
  plane        one weight per joint and sample ([n_inputs][ld_w] planes, ld_w = N + 64);
  composition  rdb_regressor_batch (and rdb_components_regressor_batch) into chunks of 2^19 samples, the rows scaled by sqrt(w) with torch,
               then G += X X^T, b += X tau by torch matmul (the plane weights).
Rates are samples per second of the median round; the weighted forms are reported relative to the unweighted call of the same chain and model.
The plane-weighted call is compared with the composition (max |a - b| over max(max |b|, 1)).  The GPU name, its power limit and the SM clock
sampled during the timed regions go with the numbers."""
import argparse
import ctypes
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rosdyn_b200 import _lib, fixtures  # noqa: E402
from bench_gram_segmented import gpu_info  # noqa: E402

CHUNK = 1 << 19


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
    assert torch.cuda.is_available(), "tools/bench_gram_weighted.py measures on a CUDA device"
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    S = a.samples
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "samples": S, "chunk_of_composition": CHUNK,
           "inputs": "device-resident: q, dq, ddq, tau_meas planes n_inputs x 2^24 doubles and weight planes (> L2)", "runs": {}}

    def timed(fn, seconds):
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
        n = d.n_inputs
        x = torch.empty((4, n, S), dtype=torch.float64, device="cuda")
        for k in range(4):
            _lib.check(lib.rdb_fill_uniform(x[k].data_ptr(), n, S, S, 0x5EED0000 + 91, k, st))
        x[3].mul_(50.0)  # measured torques in [-50, 50)
        s_all = _lib.CSamples(S, S, x[0].data_ptr(), x[1].data_ptr(), x[2].data_ptr(), None)
        tau = ctypes.c_void_p(x[3].data_ptr())
        wbuf = torch.empty((n, S + 64), dtype=torch.float64, device="cuda")
        _lib.check(lib.rdb_fill_uniform(wbuf.data_ptr(), n, S, S + 64, 0x5EED0000 + 92, 0, st))
        wbuf.add_(1.0)  # weights in [0, 2) (rdb_fill_uniform gives [-1, 1))
        weights = {"joint": _lib.CGramWeights(wbuf.data_ptr(), 1, 0), "sample": _lib.CGramWeights(wbuf.data_ptr(), 0, 1),
                   "plane": _lib.CGramWeights(wbuf.data_ptr(), S + 64, 1)}
        for model in ("rigid", "friction"):
            ch = Chain(d)
            if model == "friction":
                ch.setComponents([{"type": "friction1", "joint": j, "min_velocity": 0.05, "max_velocity": 0.7} for j in range(n)])
            ext = model == "friction"
            Pr = 10 * d.n_joints
            P = Pr + ch.getComponentColumns()
            outs = {k: torch.empty((P * P + P + 1,), dtype=torch.float64, device="cuda") for k in ("unweighted", "joint", "sample", "plane")}

            def ptrs(o):
                return [ctypes.c_void_p(o.data_ptr() + 8 * off) for off in (0, P * P, P * P + P)]

            def unweighted():
                f = lib.rdb_regressor_gram_ext_batch if ext else lib.rdb_regressor_gram_batch
                _lib.check(f(ch._h, ctypes.byref(s_all), tau, *ptrs(outs["unweighted"]), 0, st))

            def weighted(form):
                f = lib.rdb_regressor_gram_ext_weighted_batch if ext else lib.rdb_regressor_gram_weighted_batch
                return lambda: _lib.check(f(ch._h, ctypes.byref(s_all), tau, ctypes.byref(weights[form]), *ptrs(outs[form]), 0, st))

            phi = torch.empty((P * n, CHUNK), dtype=torch.float64, device="cuda")
            Gc = torch.empty((P, P), dtype=torch.float64, device="cuda")
            bc = torch.empty((P,), dtype=torch.float64, device="cuda")
            tc = torch.empty((1,), dtype=torch.float64, device="cuda")

            def composition():
                Gc.zero_(); bc.zero_(); tc.zero_()
                for lo in range(0, S, CHUNK):
                    L = min(CHUNK, S - lo)
                    s = _lib.CSamples(L, S, x[0].data_ptr() + 8 * lo, x[1].data_ptr() + 8 * lo, x[2].data_ptr() + 8 * lo, None)
                    _lib.check(lib.rdb_regressor_batch(ch._h, ctypes.byref(s), ctypes.c_void_p(phi.data_ptr()), None, CHUNK, st))
                    if ext:
                        _lib.check(lib.rdb_components_regressor_batch(ch._h, ctypes.byref(s), ctypes.c_void_p(phi.data_ptr() + 8 * Pr * n * CHUNK),
                                                                      CHUNK, st))
                    sw = wbuf[:, lo:lo + L].sqrt()
                    X = (phi[:, :L].view(P, n, L) * sw).reshape(P, n * L)
                    t = (x[3][:, lo:lo + L] * sw).reshape(n * L)
                    Gc.addmm_(X, X.T)
                    bc.addmv_(X, t)
                    tc.add_(t @ t)

            fns = {"unweighted": unweighted, "joint": weighted("joint"), "sample": weighted("sample"), "plane": weighted("plane"),
                   "composition": composition}
            for fn in fns.values():
                fn()
            torch.cuda.synchronize()
            ref = torch.cat([Gc.reshape(-1), bc, tc])
            err = float((outs["plane"] - ref).abs().max() / max(float(ref.abs().max()), 1.0))
            info = {}
            for form in ("unweighted", "plane"):
                fns[form]()
                flag = ctypes.c_int32(-1)
                buf = ctypes.create_string_buffer(512)
                lib.rdb_chain_gram_kernel_info(ch._h, ctypes.byref(flag), buf, len(buf))
                info[form] = [flag.value, buf.value.decode()[:160]]
            rounds = {k: [] for k in fns}
            clocks = []
            for _ in range(a.rounds):
                for k, fn in fns.items():
                    t, clk = timed(fn, a.seconds)
                    rounds[k].append(S / t / 1e9)
                    clocks.append(clk)
            med = {k: statistics.median(v) for k, v in rounds.items()}
            rel = {k: med[k] / med["unweighted"] for k in med}
            key = f"{name} {model}"
            res["runs"][key] = {"P": P, "G_samples_per_s": med, "vs_unweighted": rel, "rounds": rounds, "max_rel_diff_plane_vs_composition": err,
                                "kernel_info": info, "sm_mhz_median": statistics.median(c.get("sm_mhz") or 0.0 for c in clocks),
                                "throttle_reasons": sorted({r for c in clocks for r in c.get("reasons", [])})}
            print(f"{key:>12s}: " + "  ".join(f"{k} {med[k]:.4f} ({rel[k]:.3f})" for k in fns) +
                  f"  G samples/s (x unweighted); plane vs composition {err:.1e}; {res['runs'][key]['sm_mhz_median']:.0f} MHz", flush=True)
            del phi, outs
            torch.cuda.empty_cache()
        del x, wbuf
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
