"""Segmented normal equations: rdb_regressor_gram_segmented_batch, Chain.regressorGramSegmented and the C++ facade.

One call returns (G, b, tau^T tau) for every contiguous sample segment [offsets[k], offsets[k+1]) of a batch.  CPU: the entry refuses a null
chain without a device, its ctypes signature is declared, tests/cpp/gram_segmented_check.cpp compiles and links.  GPU (-m gpu): every segment
against the oracle's regressor over that segment and against rdb_regressor_gram_batch on the same samples (every test chain; empty, ragged
and multi-item segments in one call; ld > n; computed and measured torques), a segment bit for bit equal to the same samples passed alone,
the wave split (many segments, one segment longer than a wave), accumulation, tau_sq = NULL, subranges, inputs no chain joint feeds, the
residual of the nominal parameters, the general pipeline, argument errors, caller streams and the facades.
Tolerance: the suite's (assert_gram: every entry within 1e-10 of its Cauchy-Schwarz scale, maxabs <= 1e-10 * max(maxabs(ref), 1))."""
import ctypes
import os
import subprocess
import time

import numpy as np
import pytest

from conftest import CHAINS, ROOT
from rosdyn_b200 import _lib, fixtures
from test_instantiation_sweep import assert_gram, desc

ITEM = 4096  # samples per work item (32 GF_SEG_ITEM_GROUPS in csrc/gram_fused.cu)
WAVE_PER_SM = 8  # items per SM in a wave (GF_SEG_WAVE_PER_SM)
LENGTHS = [0, 1, 31, 32, 33, 1000, 3 * ITEM + 17]


def _c_call(lib, ch, s, tau, K, offs, G, b, tt, acc=0, stream=None):
    arr = None if offs is None else (ctypes.c_int64 * max(len(offs), 1))(*offs)
    return lib.rdb_regressor_gram_segmented_batch(ch, s, tau, K, arr, G, b, tt, acc, stream)


# ---------------------------------------------------------------------------------------------------------------------------------- CPU
def test_null_chain_is_refused():
    lib = _lib.load()
    s = _lib.CSamples(1, 1, None, None, None, None)
    assert _c_call(lib, None, ctypes.byref(s), None, 1, [0, 1], None, None, None) == _lib.RDB_ERR_INVALID_ARG
    assert _c_call(lib, None, None, None, 0, None, None, None, None) == _lib.RDB_ERR_INVALID_ARG


def test_ctypes_signature_is_declared():
    res, args = _lib.SYMBOLS["rdb_regressor_gram_segmented_batch"]
    assert res is ctypes.c_int32 and len(args) == 10
    assert args[3] is ctypes.c_int64 and args[4] == ctypes.POINTER(ctypes.c_int64) and args[8] is ctypes.c_int32
    assert _lib.load().rdb_regressor_gram_segmented_batch.argtypes == args


def _build_cpp(out):
    cuda = "/usr/local/cuda"
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "cpp", "gram_segmented_check.cpp"), "-o", out, "-L", os.path.join(ROOT, "rosdyn_b200"), "-lrosdyn_b200",
           "-Wl,-rpath," + os.path.join(ROOT, "rosdyn_b200"), "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(cuda, "lib64")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return out


def test_cpp_facade_compiles_and_links(tmp_path):
    exe = _build_cpp(str(tmp_path / "gram_segmented_check"))
    if _lib.load().rdb_device_count() == 0:  # without a device the binary only reports that it linked
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 0 and "compiled and linked only" in r.stdout


# ---------------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _offsets(lengths, start=0):
    return list(np.concatenate([[start], start + np.cumsum(lengths)]).astype(np.int64))


def _inputs(torch, n_in, n, seed, pad=5):
    """host arrays [n_in, n] and device views of them with plane stride n + pad (ld > n)"""
    rng = np.random.RandomState(seed)
    h = [rng.uniform(-np.pi, np.pi, (n_in, n)), rng.uniform(-2, 2, (n_in, n)), rng.uniform(-5, 5, (n_in, n)), rng.uniform(-50, 50, (n_in, n))]
    d = []
    for x in h:
        buf = torch.zeros((n_in, n + pad), dtype=torch.float64, device="cuda")
        buf[:, :n] = torch.tensor(x, device="cuda")
        d.append(buf[:, :n])
    return h, d


class SegmentReference:
    """Phi^T Phi, Phi^T tau, tau^T tau of any segment from the oracle's regressor of the whole batch (computed once)"""

    def __init__(self, d, h):
        from oracle.oracle import OracleChain
        n_in, P, n = d.n_inputs, 10 * d.n_joints, h[0].shape[1]
        phi, self.tau = OracleChain(d).regressor_torque(*h[:3], nthreads=0)
        self.X = phi.reshape(P, n_in, n)

    def __call__(self, lo, hi, tau=None):
        t = (self.tau if tau is None else tau)[:, lo:hi]
        X = self.X[:, :, lo:hi].reshape(self.X.shape[0], -1)
        return X @ X.T, X @ t.reshape(-1), float(np.sum(t * t))


def _check_segments(G, b, tt, offs, ref, tau, what):
    G, b, tt = _np(G), _np(b), _np(tt)
    for k in range(len(offs) - 1):
        lo, hi = int(offs[k]), int(offs[k + 1])
        if lo == hi:
            assert not G[k].any() and not b[k].any() and tt[k] == 0.0, f"{what}: empty segment {k} not zero"
        else:
            assert_gram(G[k], b[k], tt[k], *ref(lo, hi, tau), f"{what}: segment {k} [{lo}, {hi})")


@pytest.mark.gpu
@pytest.mark.parametrize("name", CHAINS)
def test_parity_every_chain(name, torch):
    """Segments of 0, 1, 31, 32, 33, 1 000 and 3 items + 17 samples in one call (ld > n), computed and measured torques: each against the
    oracle and against rdb_regressor_gram_batch over the same samples; a segment equals the same samples passed alone, bit for bit; two
    identical calls agree bit for bit; gramKernelInfo names the segmented kernel."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    offs = _offsets(LENGTHS)
    n = int(offs[-1])
    h, x = _inputs(torch, d.n_inputs, n, 500 + len(name))
    ref = SegmentReference(d, h)
    for tau_h, tau_d in ((None, None), (h[3], x[3])):
        what = f"{name} tau={'measured' if tau_h is not None else 'computed'}"
        G, b, tt = ch.regressorGramSegmented(*x[:3], offs, tau_meas=tau_d)
        flag, why = ch.gramKernelInfo()
        assert flag in (0, 1) and why.startswith("gram_fused_segmented_kernel, "), (flag, why)
        _check_segments(G, b, tt, offs, ref, tau_h, what)
        G2, b2, t2 = ch.regressorGramSegmented(*x[:3], offs, tau_meas=tau_d)
        assert torch.equal(G, G2) and torch.equal(b, b2) and torch.equal(tt, t2), f"{what}: two identical calls differ"
        for k in range(len(LENGTHS)):
            lo, hi = int(offs[k]), int(offs[k + 1])
            part = [v[:, lo:hi] for v in x[:3]]
            t_part = None if tau_d is None else tau_d[:, lo:hi]
            Gs, bs, ts = ch.regressorGramSegmented(*part, [0, hi - lo], tau_meas=t_part)
            assert torch.equal(Gs[0], G[k]) and torch.equal(bs[0], b[k]) and torch.equal(ts[0], tt[k]), \
                f"{what}: segment {k} differs from the same samples passed alone"
            if hi > lo:
                Go, bo, to = (_np(v) for v in ch.regressorGram(*part, tau_meas=t_part))
                assert_gram(_np(G[k]), _np(b[k]), _np(tt[k]), Go, bo, float(to[0]), f"{what}: segment {k} against rdb_regressor_gram_batch")


@pytest.mark.gpu
def test_specialised_equals_precompiled(torch, monkeypatch):
    """On an all-revolute chain the segmented kernel compiled at run time and the precompiled one agree bit for bit."""
    from rosdyn_b200.chain import Chain
    from test_gram_specialised import _both
    d = fixtures.by_name("c7")
    ch = Chain(d)
    offs = _offsets([5, 2 * ITEM + 3, 700])
    _, x = _inputs(torch, d.n_inputs, int(offs[-1]), 77)
    a, b, ia, ib = _both(ch, lambda: ch.regressorGramSegmented(*x[:3], offs), monkeypatch)
    assert ia[0] == 1 and ib[0] == 0, (ia, ib)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


@pytest.mark.gpu
def test_waves(torch, monkeypatch):
    """More segments than one wave holds (default item length and wave), and with 32-sample items and a wave of one item per SM a segment
    spread over three waves and many segments over several: every segment against the oracle."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.RandomState(9)
    many = list(rng.randint(1, 90, WAVE_PER_SM * sm + 40))  # one item each: more items than one wave holds
    h, x = _inputs(torch, d.n_inputs, int(sum(many)), 31)
    ref = SegmentReference(d, h)
    offs = _offsets(many)
    _check_segments(*ch.regressorGramSegmented(*x[:3], offs), offs, ref, None, "more segments than one wave")
    monkeypatch.setenv("RDB_GRAM_SEG_ITEM_GROUPS", "1")
    monkeypatch.setenv("RDB_GRAM_SEG_WAVE_PER_SM", "1")
    lengths = [40] * 100 + [32 * (2 * sm + 7) + 5] + [7, 0, 65] * 30  # a segment of 2 SMs + 8 items: 3 waves of its own
    h, x = _inputs(torch, d.n_inputs, int(sum(lengths)), 32)
    ref = SegmentReference(d, h)
    offs = _offsets(lengths)
    for tau_h, tau_d in ((None, None), (h[3], x[3])):
        _check_segments(*ch.regressorGramSegmented(*x[:3], offs, tau_meas=tau_d), offs, ref, tau_h, "multi-wave segment")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "random_b"])
def test_semantics(name, torch):
    """accumulate adds exactly; tau_sq = NULL is accepted; offsets covering a subrange of [0, n); the nominal parameters leave a zero residual
    tau_sq - 2 pi^T b + pi^T G pi per segment when tau = getJointTorque."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    n = 9000
    h, x = _inputs(torch, d.n_inputs, n, 41)
    ref = SegmentReference(d, h)
    offs = _offsets([100, 0, 3000, 2500], start=77)  # [77, 5677) of 9 000 samples
    G, b, tt = ch.regressorGramSegmented(*x[:3], offs, tau_meas=x[3])
    _check_segments(G, b, tt, offs, ref, h[3], f"{name} subrange")
    out = tuple(v.clone() for v in (G, b, tt))
    ch.regressorGramSegmented(*x[:3], offs, tau_meas=x[3], out=out)
    for o, v, k in zip(out, (G, b, tt), ("gram", "rhs", "tau_sq")):
        assert torch.equal(o, v + v), f"{name}: accumulated {k}"
    # tau_sq = NULL through the C-ABI
    lib = _lib.load()
    K, P = len(offs) - 1, 10 * d.n_joints
    G3, b3 = torch.full((K, P, P), np.nan, dtype=torch.float64, device="cuda"), torch.full((K, P), np.nan, dtype=torch.float64, device="cuda")
    s = ch._samples(n, list(x[:3]) + [None])
    torch.cuda.synchronize()
    assert _c_call(lib, ch._h, ctypes.byref(s), ctypes.c_void_p(x[3].data_ptr()), K, offs, ctypes.c_void_p(G3.data_ptr()),
                   ctypes.c_void_p(b3.data_ptr()), None) == _lib.RDB_OK
    torch.cuda.synchronize()
    assert torch.equal(G3, G) and torch.equal(b3, b), f"{name}: tau_sq = NULL changed gram / rhs"
    # residual of the nominal parameters with the computed torque
    G, b, tt = (_np(v) for v in ch.regressorGramSegmented(*x[:3], offs))
    pi = ch.getNominalParameters()
    for k in range(K):
        if offs[k + 1] > offs[k]:
            res = tt[k] - 2.0 * pi @ b[k] + pi @ G[k] @ pi
            assert abs(res) <= 1e-9 * tt[k], f"{name}: segment {k} residual {res:.3e} of tau_sq {tt[k]:.3e}"


@pytest.mark.gpu
def test_unfed_input_with_measured_torque(torch):
    """An input no chain joint feeds, with measured torques: each segment's tau_sq includes that input's squares."""
    from rosdyn_b200.chain import Chain
    d = desc("k3_rev_unfed_input")
    ch = Chain(d)
    offs = _offsets([0, 1, 33, 1000, 2 * ITEM + 1])
    h, x = _inputs(torch, d.n_inputs, int(offs[-1]), 51)
    ref = SegmentReference(d, h)
    _check_segments(*ch.regressorGramSegmented(*x[:3], offs, tau_meas=x[3]), offs, ref, h[3], "unfed input")
    _check_segments(*ch.regressorGramSegmented(*x[:3], offs), offs, ref, None, "unfed input, computed torque")
    out = tuple(v.clone() for v in ch.regressorGramSegmented(*x[:3], offs, tau_meas=x[3]))
    first = tuple(v.clone() for v in out)
    ch.regressorGramSegmented(*x[:3], offs, tau_meas=x[3], out=out)
    for o, v in zip(out, first):
        assert torch.equal(o, v + v)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["generic12", "k0_no_moving_joint"])
def test_general_pipeline(name, torch):
    """Chains outside the fused kernel run the general pipeline once per segment, and gramKernelInfo says so."""
    from rosdyn_b200.chain import Chain
    d = fixtures.random_chain(1212, 12, p_fixed=0.0) if name == "generic12" else desc(name)
    ch = Chain(d)
    offs = _offsets([0, 1, 33, 1000, 1500])
    h, x = _inputs(torch, d.n_inputs, int(offs[-1]), 61)
    ref = SegmentReference(d, h)
    for tau_h, tau_d in ((None, None), (h[3], x[3])):
        _check_segments(*ch.regressorGramSegmented(*x[:3], offs, tau_meas=tau_d), offs, ref, tau_h, name)
        flag, why = ch.gramKernelInfo()
        assert flag == 2 and why.startswith("general pipeline: one pass per segment"), (flag, why)


@pytest.mark.gpu
def test_argument_errors(torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    lib = _lib.load()
    n, P = 100, 60
    _, x = _inputs(torch, 6, n, 71)
    G = torch.zeros((3, P, P), dtype=torch.float64, device="cuda")
    b = torch.zeros((3, P), dtype=torch.float64, device="cuda")
    tt = torch.zeros((3,), dtype=torch.float64, device="cuda")
    pG, pb, pt = (ctypes.c_void_p(v.data_ptr()) for v in (G, b, tt))
    s = ch._samples(n, list(x[:3]) + [None])
    bad = {"n_segments < 0": (-1, [0]), "offsets NULL": (2, None), "decreasing": (2, [0, 50, 20]), "negative start": (2, [-1, 5, 9]),
           "past n": (2, [0, 50, n + 1])}
    for what, (K, offs) in bad.items():
        assert _c_call(lib, ch._h, ctypes.byref(s), None, K, offs, pG, pb, pt) == _lib.RDB_ERR_INVALID_ARG, what
        assert lib.rdb_last_error().decode(), what
    assert _c_call(lib, ch._h, ctypes.byref(s), None, 2, [0, 5, 9], None, pb, pt) == _lib.RDB_ERR_INVALID_ARG
    assert _c_call(lib, ch._h, ctypes.byref(s), None, 2, [0, 5, 9], pG, None, pt) == _lib.RDB_ERR_INVALID_ARG
    s2 = ch._samples(n, [x[0], None, x[2], None])
    assert _c_call(lib, ch._h, ctypes.byref(s2), None, 2, [0, 5, 9], pG, pb, pt) == _lib.RDB_ERR_DIM_MISMATCH
    assert _c_call(lib, ch._h, ctypes.byref(s), None, 0, None, None, None, None) == _lib.RDB_OK
    torch.cuda.synchronize()
    assert not G.any() and not b.any() and not tt.any(), "a refused call wrote"
    with pytest.raises(ValueError):
        ch.regressorGramSegmented(*(_np(v) for v in x[:3]), [0, n])
    with pytest.raises(_lib.RosdynB200Error):
        ch.regressorGramSegmented(*x[:3], [0, 50, 20])


@pytest.mark.gpu
def test_streams(torch):
    """On a caller stream the entry equals its default-stream result bit for bit, and it is ordered after an rdb_regressor_gram_batch of the
    same handle issued on another stream (that one waits behind a gate)."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    offs = _offsets([300, 0, ITEM + 1, 50])
    _, x = _inputs(torch, d.n_inputs, int(offs[-1]), 81)
    solo = ch.regressorGramSegmented(*x[:3], offs)
    big = [v.repeat(1, 64).contiguous() for v in x[:3]]
    g_solo = ch.regressorGram(*big)  # also compiles the unsegmented kernel before the gate starts
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    done1, done2 = torch.cuda.Event(), torch.cuda.Event()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(2_000_000_000)  # about a second at the SM clock
        g1 = ch.regressorGram(*big)
        done1.record()
    with torch.cuda.stream(s2):
        seg = ch.regressorGramSegmented(*x[:3], offs)
        done2.record()
    time.sleep(0.2)
    assert not done1.query() and not done2.query(), "the segmented call on the second stream did not wait for the first stream's Gram call"
    torch.cuda.synchronize()
    for u, v in zip(seg, solo):
        assert torch.equal(u, v)
    for u, v in zip(g1, g_solo):
        assert torch.equal(u, v)


@pytest.mark.gpu
def test_facades(torch, tmp_path):
    """The C++ facade program runs; the Python method returns G[K,P,P], b[K,P], tau_sq[K] as CUDA float64 tensors."""
    exe = _build_cpp(str(tmp_path / "gram_segmented_check"))
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "segmented gram facade ok" in r.stdout, r.stdout + r.stderr
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c7")
    ch = Chain(d)
    _, x = _inputs(torch, d.n_inputs, 500, 91)
    G, b, tt = ch.regressorGramSegmented(*x[:3], [0, 100, 100, 500])
    for t, shape in ((G, (3, 70, 70)), (b, (3, 70)), (tt, (3,))):
        assert tuple(t.shape) == shape and t.is_cuda and t.dtype == torch.float64
