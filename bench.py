#!/usr/bin/env python
"""bench.py - headline benchmark of the rosdyn::Chain hot path on B200 (BASELINE.json metric:
"6-DOF regressor+torque samples/sec (fp64)").

One step = one pass of the hot path over one batch of synthetic (q,Dq,DDq) samples of the UR10-like 6-DOF chain
(C6, SURVEY.md section 8d): getRegressor + getJointTorque for every sample.

  --workload materialise : Phi (6x70, 420 SoA planes) + tau (6 planes) written to HBM        (HBM roofline)
  --workload gram        : Phi and tau consumed in-kernel by the normal equations Phi^T Phi / Phi^T tau
                           (FP64 DMMA roofline); N>1 adds one NCCL all-reduce of the (70^2+70+1) partials per step

`value`  : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`    : the same metric through the C-ABI host-buffer entry point (pinned host inputs, H2D/D2H inside the timed region).
`--impl reference` : the reference's CPU Chain loop on all host threads.  Two builds of it exist under oracle/: the plain-C restatement
                     (kind "port") and oracle/_ref, the reference's own headers compiled against stand-in Eigen/urdf/ros headers (kind
                     "reference"; its dense arithmetic is the stand-in's plain loops, so it is the slower of the two).  Both are timed; the
                     line's value is the FASTER one (the conservative baseline), the other is reported beside it.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "6-DOF regressor+torque samples/sec (fp64)"
UNIT = "samples/s"
SEED = 0x5EED0000 + 1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("RDB_BENCH_WORKLOAD", "gram"), choices=["materialise", "gram"])
    ap.add_argument("--chain", default="c6")
    ap.add_argument("--samples", type=int, default=0, help="samples per step per GPU (0 = workload default)")
    ap.add_argument("--e2e-samples", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target length of the bounded CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--pageable", action="store_true", help="e2e leg with pageable (malloc) host buffers instead of pinned ones")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (gram: gram, rhs, tau_sq; "
                         "materialise: a fixed, seeded sample of the columns of regressor and torque of the last launch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours: the CPU timing loop does not store its outputs")
    return args


DUMP_COLUMNS = 8192   # materialise: sampled columns of Phi / tau written by --dump-outputs (426 rows x 8 B x 8192 = 28 MB for C6)


def dump_outputs(path: str, arrays: dict):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), t.detach().cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons during the timed region (NVML; nvidia-smi fallback)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    p = self._nvml
                    self.samples.append(float(p.nvmlDeviceGetClockInfo(self._h, p.NVML_CLOCK_SM)))
                    r = p.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(p, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else p.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    table = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                             "hw_power_brake_slowdown": 0x80}
                    for k, bit in table.items():
                        if r & bit:
                            self.reasons.add(k)
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                    self.samples.append(float(out[0]))
                    self.max_mhz = float(out[1])
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=2)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def ncu_traffic_per_sample(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per sample of the named kernel, from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py); None when there is no capture for it."""
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[kernel]["dram_bytes_per_sample"])
    except Exception:
        return None


def sass_counts(key: str):
    """FP64 instructions of the named kernel counted in its SASS (profiles/gram_fused_sass.json, written by tools/sass_counts.py at build time
    from the cubin that ships): {"gen_dp_instr_per_sample": .., "gen_flop_per_sample": .., "dmma_per_4_samples": ..}; None when absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "gram_fused_sass.json")))[key]
    except Exception:
        return None


def h2d_probe(dev, world, nbytes=1 << 30, reps=3):
    """Bare pinned-host -> device cudaMemcpyAsync bandwidth of this rank while ALL ranks copy at the same time (GB/s): the ceiling of any
    end-to-end number on this box (PCIe link per GPU at N = 1; host memory / PCIe fabric shared by the ranks at N > 1)."""
    import torch
    import torch.distributed as dist
    src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    src.fill_(1)
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    gbs = reps * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    t = torch.tensor([gbs], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return float(t[0])


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_run(chain_name: str, n: int, threads: int, reps: int = 1, kind="port"):
    """getJointTorque + getRegressor per sample on the CPU, all samples resident in host memory.
    kind "port": the plain-C restatement (oracle/rosdyn_oracle.c); "reference": the reference's own rosdyn::Chain (oracle/_ref)."""
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200 import fixtures
    d = fixtures.by_name(chain_name)
    oc = OracleChain(d, fast="ref" if kind == "reference" else False)
    q, dq, ddq = (fill_uniform(d.n_inputs, n, SEED, s) for s in range(3))
    best = None
    for _ in range(reps):
        t = time.perf_counter()
        oc.regressor_torque(q, dq, ddq, nthreads=threads, store=False)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return n / best, best


def host_threads() -> int:
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1, so do not ask OpenMP)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def reference_build_rate(chain_name: str, seconds: float, threads: int):
    """The reference's own headers (oracle/_ref) on the same workload; None when that build is absent."""
    try:
        from oracle import oracle
        if not oracle.have_ref():
            return None
        rate, _ = cpu_run(chain_name, 2000 * threads, threads, kind="reference")
        n = int(max(2000 * threads, min(rate * seconds, 5_000_000)))
        rate, dt = cpu_run(chain_name, n, threads, kind="reference")
        return {"value": rate, "unit": UNIT, "cores": threads, "kind": "reference",
                "sample": f"{n} samples, rosdyn::Chain::getJointTorque + getRegressor of the reference's own headers compiled against the "
                          f"stand-in Eigen of oracle/shim (one Chain::clone() per thread, OpenMP {threads} threads, {dt:.1f} s)"}
    except Exception as e:  # the checker build must never take the bench down
        return {"unavailable": repr(e)}


def cpu_baseline(chain_name: str, seconds: float):
    threads = host_threads()
    rate, _ = cpu_run(chain_name, 20000 * max(1, threads // 4), threads)       # calibration
    n = int(max(50_000, min(rate * seconds, 50_000_000)))
    rate, dt = cpu_run(chain_name, n, threads)
    out = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": f"{n} samples of the same workload (getJointTorque + getRegressor per sample, oracle/rosdyn_oracle.c, "
                     f"OpenMP {threads} threads, {dt:.1f} s)"}
    ref = reference_build_rate(chain_name, min(4.0, seconds), threads)
    if ref is not None:
        out["reference_build"] = ref   # slower than the port (plain-loop stand-in for Eigen): the port stays the baseline
    return out


def run_reference(args):
    """--impl reference: the reference's CPU Chain loop on all host threads (the faster of the restatement and oracle/_ref)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    rate, _ = cpu_run(args.chain, 20000 * max(1, threads // 4), threads)
    n = int(max(20_000, min(rate * 4.0, 20_000_000)))                           # ~4 s per step
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200 import fixtures
    d = fixtures.by_name(args.chain)
    oc = OracleChain(d)
    q, dq, ddq = (fill_uniform(d.n_inputs, n, SEED, s) for s in range(3))
    for _ in range(min(args.warmup, 1)):
        oc.regressor_torque(q, dq, ddq, nthreads=threads, store=False)
    t = time.perf_counter()
    for _ in range(args.steps):
        oc.regressor_torque(q, dq, ddq, nthreads=threads, store=False)
    dt = time.perf_counter() - t
    v = n * args.steps / dt
    ref = reference_build_rate(args.chain, 4.0, threads)
    kind, note = "port", "oracle/rosdyn_oracle.c (plain-C restatement of primitives_impl.h), OpenMP"
    if ref and ref.get("value", 0.0) > v:   # report the faster CPU build: the conservative baseline
        v, kind, note = ref["value"], "reference", ref["sample"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"{d.name}: getRegressor (6x70) + getJointTorque per sample (the GPU arm's workload), evaluated by the CPU "
                               f"restatement of the reference's Chain loop; bounded sample of {n} samples/step",
                   "chain": d.name, "samples_per_step": n, "mode": args.workload},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{n} samples/step x {args.steps} steps, {note}", "reference_build": ref},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def bind_to_gpu_numa_node(index: int):
    """Pin this rank to the CPUs NVML reports as local to its GPU, so that the pinned host buffers of the e2e leg are first-touched on the
    GPU's NUMA node (8 ranks reading from one socket do not reach 8 x PCIe bandwidth).  Returns the previous affinity (restored before
    the CPU baseline leg) or None when NVML / the syscall is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        old = os.sched_getaffinity(0)
        cpus &= old
        if cpus:
            os.sched_setaffinity(0, cpus)
            return old
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import ctypes

    import torch
    import torch.distributed as dist
    from rosdyn_b200 import fixtures
    from rosdyn_b200._lib import CSamples, check, load
    from rosdyn_b200.chain import Chain, fill_uniform, fp64_peak, kernel_launch_count
    from rosdyn_b200.sharding import Group

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    old_affinity = bind_to_gpu_numa_node(local) if world > 1 else None
    # rank 0 prints ONE JSON line on stdout: everything else that lands on file descriptor 1 from here on (NCCL prints its version banner
    # there) is sent to stderr, and the JSON line goes to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    d = fixtures.by_name(args.chain)
    lib = load()
    n_in, P = d.n_inputs, 10 * d.n_joints
    gram = args.workload == "gram"
    # Samples per GPU per step.  gram: 128 M samples = 18.4 GB of device-resident inputs, ~73 ms per step, so the driver's 20 steps give a
    # timed region of ~1.5 s under sustained clocks / power (round 1 timed 8 M samples per step: 0.1 s of burst clocks).  materialise: a step
    # is `launches` back-to-back launches of 4 M samples each over DISTINCT inputs (128 M samples per step: ~75 ms); Phi (13.6 GB per launch)
    # is overwritten in place.
    if gram:
        S, launches = (args.samples or 128_000_000), 1
        Sl = S
    else:
        Sl = 4_000_000
        launches = max(1, (args.samples or 128_000_000) // Sl)
        S = Sl * launches
    # weak scaling: every rank owns its own shard of S samples (disjoint sample indices via the seed offset)
    q, dq, ddq = (fill_uniform(n_in, S, SEED + 1000003 * rank, s, device=dev) for s in range(3))
    if gram:
        # N > 1: the C-ABI's NCCL group (rdb_group_create_rank): fused kernel -> packed partials -> ncclAllReduce -> caller's arrays, all on
        # one stream below the C-ABI; torch.distributed only carries the 128-byte NCCL id and the barriers
        grp = Group.from_torch_distributed(d, local)
        ch_h = ctypes.c_void_p(lib.rdb_group_chain(grp._h, 0))
        G = torch.zeros((P, P), dtype=torch.float64, device=dev)
        b = torch.zeros((P,), dtype=torch.float64, device=dev)
        tt = torch.zeros((1,), dtype=torch.float64, device=dev)
        out = [(G, b, tt)]
        shards = [(q, dq, ddq)]
    else:
        ch = Chain(d)
        ch_h = ch._h
        phi = torch.empty((P * n_in, Sl), dtype=torch.float64, device=dev)
        tau = torch.empty((n_in, Sl), dtype=torch.float64, device=dev)
        smps = [CSamples(Sl, S, q[:, k * Sl:].data_ptr(), dq[:, k * Sl:].data_ptr(), ddq[:, k * Sl:].data_ptr(), None) for k in range(launches)]

    def step():
        if gram:
            grp.gram(shards, out=out)     # rdb_regressor_gram_sharded on torch's current stream (one rank: no collective)
        else:
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for smp in smps:
                check(lib.rdb_regressor_batch(ch_h, ctypes.byref(smp), phi.data_ptr(), tau.data_ptr(), Sl, st))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    l0 = kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches_timed = kernel_launch_count() - l0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    value = world * S * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        if gram:
            dump_outputs(args.dump_outputs, {"gram": G, "rhs": b, "tau_sq": tt})
        else:   # Phi / tau hold the last launch of the last step; the sampled columns depend only on the launch size
            import numpy as np
            cols = np.sort(np.random.default_rng(0).choice(Sl, size=min(Sl, DUMP_COLUMNS), replace=False))
            cols = torch.from_numpy(cols).to(dev)
            dump_outputs(args.dump_outputs, {"regressor": phi.index_select(1, cols), "torque": tau.index_select(1, cols)})

    # ------------------------------------------------------------------ e2e through the host-buffer C-ABI entry
    e2e = None
    if not args.no_e2e:
        probe = h2d_probe(dev, world)
        Se = args.e2e_samples or (16_000_000 if gram else 500_000)

        def host_buf(rows, cols):
            t_ = torch.empty((rows, cols), dtype=torch.float64)
            return t_ if args.pageable else t_.pin_memory()
        hq, hdq, hddq = (host_buf(n_in, Se) for _ in range(3))
        for k, h in enumerate((hq, hdq, hddq)):
            lib.rdb_fill_uniform_host(h.data_ptr(), n_in, Se, Se, SEED + 1000003 * rank, k)
        hs = CSamples(Se, Se, hq.data_ptr(), hdq.data_ptr(), hddq.data_ptr(), None)
        if gram:
            hG, hb, ht = host_buf(P, P), host_buf(1, P), host_buf(1, 1)
            dflat = torch.empty((P * P + P + 1,), dtype=torch.float64, device=dev)
            hflat = torch.empty((P * P + P + 1,), dtype=torch.float64).pin_memory()

            def e2e_step():
                check(lib.rdb_regressor_gram_batch_host(ch_h, ctypes.byref(hs), None, hG.data_ptr(), hb.data_ptr(), ht.data_ptr(), 0))
                if world > 1:   # the partials of the ranks are summed over NVLink and read back
                    hflat[:P * P] = hG.reshape(-1)
                    hflat[P * P:P * P + P] = hb.reshape(-1)
                    hflat[P * P + P:] = ht.reshape(-1)
                    dflat.copy_(hflat, non_blocking=True)
                    dist.all_reduce(dflat)
                    hflat.copy_(dflat)
            h2d, d2h = 3 * n_in * Se * 8, (P * P + P + 1) * 8
        else:
            hphi, htau = host_buf(P * n_in, Se), host_buf(n_in, Se)

            def e2e_step():
                check(lib.rdb_regressor_batch_host(ch_h, ctypes.byref(hs), hphi.data_ptr(), htau.data_ptr(), Se))
            h2d, d2h = 3 * n_in * Se * 8, (P * n_in + n_in) * Se * 8
        for _ in range(2):
            e2e_step()
        ke = max(2, min(args.steps, 5))
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            e2e_step()
        barrier()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        sec = float(te[0])
        link_gbs = (h2d + d2h) * ke / sec / 1e9       # bytes this rank moved over its PCIe link per second
        e2e = {"value": world * Se * ke / sec, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "samples_per_step_per_gpu": Se, "steps": ke, "host_buffers": "pageable" if args.pageable else "pinned",
               "api": "rdb_regressor_gram_batch_host" if gram else "rdb_regressor_batch_host",
               "link_GBps_per_gpu": link_gbs, "h2d_probe_GBps_per_gpu": probe, "frac_of_h2d": link_gbs / probe if probe else None,
               "probe": "bare pinned cudaMemcpyAsync H2D of 1 GiB x 3 on every rank at the same time (min over ranks): the box's ceiling"}

    # ------------------------------------------------------------------ roofline of the dominant kernel
    peaks, src = measured_peaks()
    per_launch_s = ms * 1e-3 / args.steps / launches
    if gram:
        # algorithmic FLOPs per sample, BLAS SYRK+GEMV convention (SURVEY.md 8d): n_act*P*(P+1) + 2*n_act*P
        flop = n_in * P * (P + 1) + 2 * n_in * P
        peak, peaks64 = None, None
        if rank == 0:
            peaks64 = {"dmma_m8n8k4": fp64_peak("dmma", 3), "dfma": fp64_peak("dfma", 3), "dmma_and_dfma_interleaved": fp64_peak("mixed", 3)}
            peak = max(peaks64["dmma_m8n8k4"], peaks64["dfma"])
        ach = Sl * flop / per_launch_s / 1e12
        K = sum(1 for j in d.joints if j.input_index >= 0)
        tps = ncu_traffic_per_sample(f"gram_fused_kernel<{d.n_joints}>:{args.chain}")
        # What the kernel executes (counted in the SASS of the cubin that ships, tools/sass_counts.py): per sample, DMMA m8n8k4 tiles of the
        # folded, structurally non-zero part of the augmented Gram matrix (512 flop each, 4 samples per tile) and the FP64 instructions of the
        # regressor generation (DFMA = 2 flop, DMUL / DADD = 1 flop).  Both share ONE FP64 datapath: a DMMA holds it 16 cycles, any other FP64
        # warp instruction 2 cycles, so `datapath_busy_frac` = (16 * DMMA + 2 * FP64 instr) per sample / available datapath cycles per sample.
        rev = all(j.type == 1 for j in d.joints if j.input_index >= 0)
        sc = sass_counts(f"K{K}_{'rev' if rev else 'gen'}") or {}
        sps = Sl / per_launch_s
        dmma4 = sc.get("dmma_per_4_samples")
        ex = None
        if dmma4 is not None and peak:
            dmma_flop = dmma4 * 512 / 4
            gen_flop = sc.get("gen_flop_per_sample", 0.0)
            gen_instr = sc.get("gen_dp_instr_per_sample", 0.0)
            sm_clock = (clk.summary()["sm_mhz"] or 1965.0) * 1e6
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
            cycles_avail = n_sm * 4 * sm_clock / sps                       # FP64-datapath cycles (one datapath per SM sub-partition) per sample
            cycles_used = 16.0 * dmma4 / 4 + 2.0 * gen_instr / 32     # a generator warp instruction serves 32 samples
            ex = {"moving_joints": K, "dmma_per_4_samples": dmma4, "dmma_flop_per_sample": dmma_flop, "generation_flop_per_sample": gen_flop,
                  "generation_fp64_instr_per_sample": gen_instr, "executed_tflops": sps * (dmma_flop + gen_flop) / 1e12,
                  "executed_flop_frac": sps * (dmma_flop + gen_flop) / 1e12 / peak,
                  "dmma_frac_of_peak": sps * dmma_flop / 1e12 / peak,
                  "datapath_busy_frac": cycles_used / cycles_avail,
                  "note": "achieved/frac use the ALGORITHMIC flops of the reference's dense n_act x 10nJ regressor (SYRK+GEMV convention, SURVEY.md 8d); "
                          "structural zeros and rigidly attached links are not multiplied, so frac can exceed 1.  executed_* count what the kernel "
                          "really issues (DMMA tiles + regressor generation); datapath_busy_frac is their occupancy of the FP64 datapath at the "
                          "SM clock sampled during the run."}
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if peak else None,
                "traffic": (tps * Sl) if tps else None,
                "peak_source": "own FP64 micro-benchmark on this GPU (max of DMMA m8n8k4 and DFMA); MEASURED_PEAKS.json has no FP64 figure",
                "fp64_peaks_tflops": peaks64, "flop_per_sample": flop, "executed": ex,
                "kernel": (sc.get("kernel") or f"gram_fused_kernel<{K},...>") + " on the folded chain (regressor generation + DMMA normal equations)"}
    else:
        bytes_per_sample = 8 * (3 * n_in + P * n_in + n_in)          # 3552 B for C6 (SURVEY.md 8d)
        ach = Sl * bytes_per_sample / per_launch_s / 1e9
        peak = float(peaks["hbm_gbs"])
        tps = ncu_traffic_per_sample(f"dyn_kernel<{d.n_joints},3>:{args.chain}")
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": (tps * Sl) if tps else None,
                "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({src})", "bytes_per_sample": bytes_per_sample, "kernel": f"dyn_kernel<{d.n_joints},3> (regressor+torque)"}

    if old_affinity is not None:
        os.sched_setaffinity(0, old_affinity)
    if rank == 0:
        cpu = None if args.no_cpu_baseline else cpu_baseline(args.chain, args.cpu_seconds)
        out_line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": (f"{d.name}: getRegressor ({n_in}x{P}) + getJointTorque per sample, "
                                    + ("fused into Phi^T Phi / Phi^T tau normal equations" if gram else f"materialised as {P * n_in + n_in} SoA planes in HBM")),
                       "chain": d.name, "samples_per_step_per_gpu": S, "launches_per_step": launches, "mode": args.workload,
                       "timed_region_s": ms * 1e-3,
                       "l2": "inputs (and outputs) per launch are far larger than the 126 MB L2; no flush needed",
                       "parallelism": f"{world} x independent sample shards" + (" + one ncclAllReduce of the partials inside the C-ABI group (rdb_regressor_gram_sharded)" if gram and world > 1 else "")},
            "e2e": e2e, "gpu_launches": int(launches_timed), "roofline": roof, "cpu_baseline": cpu, "clocks": clk.summary(),
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(out_line) + "\n").encode())
    if gram:
        del grp
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
