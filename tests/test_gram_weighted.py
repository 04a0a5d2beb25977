"""Weighted normal equations: rdb_regressor_gram_weighted_batch, rdb_regressor_gram_ext_weighted_batch, the `weights=` keyword of
Chain.regressorGram / regressorGramExt and the C++ facade overloads.

  G = sum_s Phi_s^T W_s Phi_s,  b = sum_s Phi_s^T W_s tau_s,  tau_sq = sum_s tau_s^T W_s tau_s,  W_s = diag(w[r, s])

CPU: null chain, null weights and negative strides are refused; the ctypes signatures are declared; tests/cpp/gram_weighted_check.cpp compiles
and links; the run-time specialised weighted C6 / C7 cubins build (NVRTC, host only).  GPU (-m gpu): every test chain, folded chains and the
general pipeline against the oracle's regressor contracted with the weights in numpy, in all four weight forms, computed and measured
torques, past the first reuse of the slots with a ragged tail; the extended model for XC = 2, 4, 8; w == 1 bit for bit equal to the
unweighted entries on every kernel path, and w == 4, 1/4 exactly 4x, 1/4x; one-hot per-joint weights; sample masks; inputs no chain joint
feeds; accuracy at 10^6 samples; the OLS -> per-joint sigma -> WLS loop; reproducibility, accumulate, tau_sq = NULL, caller streams, the
kernel info and the facades.  Tolerance: the suite's assert_gram."""
import ctypes
import os
import subprocess
import time

import numpy as np
import pytest

from conftest import CHAINS, ROOT
from rosdyn_b200 import _lib, fixtures
from test_instantiation_sweep import assert_gram, components, desc

N_REUSE = 20_011  # past 18 944 = 148 SMs x 4 slots x 32 samples, where the slots are first reused; not a multiple of 32
FORMS = ("joint", "sample", "plane", "scalar")


def _c_call(lib, ch, s, tau, w, G, b, tt, acc=0, stream=None, ext=False):
    f = lib.rdb_regressor_gram_ext_weighted_batch if ext else lib.rdb_regressor_gram_weighted_batch
    return f(ch, s, tau, w, G, b, tt, acc, stream)


# ---------------------------------------------------------------------------------------------------------------------------------- CPU
def test_argument_errors_without_device():
    """Null weights, a null weight pointer and negative strides are refused first, then a null chain, before anything touches a device."""
    lib = _lib.load()
    s = _lib.CSamples(1, 1, None, None, None, None)
    buf = (ctypes.c_double * 4)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    bad = {"null weights": None, "null w": ctypes.byref(_lib.CGramWeights(None, 1, 0)),
           "negative joint stride": ctypes.byref(_lib.CGramWeights(p, -1, 0)), "negative sample stride": ctypes.byref(_lib.CGramWeights(p, 0, -1))}
    for ext in (False, True):
        for what, w in bad.items():
            assert _c_call(lib, None, ctypes.byref(s), None, w, p, p, p, ext=ext) == _lib.RDB_ERR_INVALID_ARG, what
            assert "weight" in lib.rdb_last_error().decode(), what
        good = ctypes.byref(_lib.CGramWeights(p, 1, 0))
        assert _c_call(lib, None, ctypes.byref(s), None, good, p, p, p, ext=ext) == _lib.RDB_ERR_INVALID_ARG
        assert "null chain" in lib.rdb_last_error().decode()


def test_ctypes_signatures_are_declared():
    lib = _lib.load()
    for name in ("rdb_regressor_gram_weighted_batch", "rdb_regressor_gram_ext_weighted_batch"):
        res, args = _lib.SYMBOLS[name]
        assert res is ctypes.c_int32 and len(args) == 9, name
        assert args[3] == ctypes.POINTER(_lib.CGramWeights) and args[7] is ctypes.c_int32, name
        assert getattr(lib, name).argtypes == args
    assert [f[0] for f in _lib.CGramWeights._fields_] == ["w", "joint_stride", "sample_stride"]
    assert ctypes.sizeof(_lib.CGramWeights) == 24


def _build_cpp(out):
    cuda = "/usr/local/cuda"
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "cpp", "gram_weighted_check.cpp"), "-o", out, "-L", os.path.join(ROOT, "rosdyn_b200"), "-lrosdyn_b200",
           "-Wl,-rpath," + os.path.join(ROOT, "rosdyn_b200"), "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(cuda, "lib64")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return out


def test_cpp_facade_compiles_and_links(tmp_path):
    exe = _build_cpp(str(tmp_path / "gram_weighted_check"))
    if _lib.load().rdb_device_count() == 0:
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 0 and "compiled and linked only" in r.stdout


@pytest.mark.parametrize("name,args", [("c6", "gram_fused_weighted_kernel<6, 4, true, 0"), ("c7", "gram_fused_weighted_kernel<7, 3, true, 0"),
                                       ("c6", "gram_fused_weighted_kernel<6, 3, true, 2"), ("c7", "gram_fused_weighted_kernel<7, 3, true, 2"),
                                       ("c6", "gram_fused_weighted_kernel<6, 3, true, 8"), ("c7", "gram_fused_weighted_kernel<7, 2, true, 8")])
def test_specialised_cubin_builds(name, args, tmp_path):
    """NVRTC builds the weighted rigid and extended kernels against the C6 / C7 constants (host only; skipped without NVRTC)."""
    from rosdyn_b200.descriptor import to_ctypes
    lib = _lib.load()
    cdesc, keep = to_ctypes(fixtures.by_name(name))
    path = str(tmp_path / "k.cubin")
    why = ctypes.create_string_buffer(4096)
    st = lib.rdb_gram_specialised_cubin(ctypes.byref(cdesc), args.encode(), b"sm_100a", path.encode(), why, len(why))
    if st != _lib.RDB_OK and "NVRTC not found" in why.value.decode():
        pytest.skip(why.value.decode())
    assert st == _lib.RDB_OK, why.value.decode()
    assert os.path.getsize(path) > 10_000


# ---------------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _inputs(torch, n_in, n, seed, pad=5):
    """host arrays [n_in, n] (q, dq, ddq, tau) and device views of them with plane stride n + pad (ld > n)"""
    rng = np.random.RandomState(seed)
    h = [rng.uniform(-np.pi, np.pi, (n_in, n)), rng.uniform(-2, 2, (n_in, n)), rng.uniform(-5, 5, (n_in, n)), rng.uniform(-50, 50, (n_in, n))]
    d = []
    for x in h:
        buf = torch.zeros((n_in, n + pad), dtype=torch.float64, device="cuda")
        buf[:, :n] = torch.tensor(x, device="cuda")
        d.append(buf[:, :n])
    return h, d


def _weights(torch, form, n_in, n, seed):
    """(host weights broadcast to [n_in, n], the device tensor of that form).  plane: rows of stride n + 11 (neither ld nor n)."""
    rng = np.random.RandomState(seed)
    if form == "joint":
        w = rng.uniform(0.01, 4.0, n_in)
        return np.broadcast_to(w[:, None], (n_in, n)), torch.tensor(w, device="cuda")
    if form == "sample":
        w = rng.uniform(0.0, 3.0, n)
        w[rng.rand(n) < 0.1] = 0.0  # masked samples
        return np.broadcast_to(w[None, :], (n_in, n)), torch.tensor(w, device="cuda")
    if form == "plane":
        w = rng.uniform(0.0, 2.0, (n_in, n))
        buf = torch.zeros((n_in, n + 11), dtype=torch.float64, device="cuda")
        buf[:, :n] = torch.tensor(w, device="cuda")
        return w, buf[:, :n]
    w = float(rng.uniform(0.5, 2.0))
    return np.full((n_in, n), w), torch.tensor(w, dtype=torch.float64, device="cuda")


class Reference:
    """The oracle's regressor of a batch ([Phi | Phi_c] with components) contracted with weights in numpy, in slices of samples"""

    def __init__(self, d, h, comps=None):
        from oracle import oracle
        from oracle.oracle import OracleChain
        n_in, P, n = d.n_inputs, 10 * d.n_joints, h[0].shape[1]
        phi, self.tau = OracleChain(d).regressor_torque(*h[:3], nthreads=0)
        X = phi.reshape(P, n_in, n)
        if comps:
            pc = sum(3 if t == 2 else 2 for t, _, _, _ in comps)
            X = np.concatenate([X, oracle.components_regressor(comps, n_in, h[0], h[1]).reshape(pc, n_in, n)])
        self.X = X

    def __call__(self, w, tau=None, lo=0, hi=None, step=16384):
        t = self.tau if tau is None else tau
        hi = self.X.shape[2] if hi is None else hi
        P = self.X.shape[0]
        G, b, tt = np.zeros((P, P)), np.zeros(P), 0.0
        for a in range(lo, hi, step):
            e = min(a + step, hi)
            X, ws, ts = self.X[:, :, a:e], w[:, a:e], t[:, a:e]
            Xw = (X * ws[None]).reshape(P, -1)
            G += Xw @ X.reshape(P, -1).T
            b += Xw @ ts.reshape(-1)
            tt += float(np.sum(ws * ts * ts))
        return G, b, tt


def _check(out, ref, what):
    G, b, tt = (_np(v) for v in out)
    assert_gram(G, b, tt, *ref, what)


def _equal(torch, a, b, what):
    for u, v, k in zip(a, b, ("gram", "rhs", "tau_sq")):
        assert torch.equal(u, v), f"{what}: {k} differs"


def _general12():
    return fixtures.random_chain(1212, 12, p_fixed=0.0)


PARITY_CHAINS = CHAINS + ["fold4_rev_tool", "fold6_mix_plain", "fold9_rev_plain", "generic12"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", PARITY_CHAINS)
def test_parity_every_chain(name, torch):
    """The four weight forms, computed and measured torques, 20 011 samples (ld > n, ragged tail) against the oracle; the kernel info
    names the weighted kernel on the fused path and the general pipeline elsewhere."""
    from rosdyn_b200.chain import Chain
    d = _general12() if name == "generic12" else (fixtures.by_name(name) if name in CHAINS else desc(name))
    ch = Chain(d)
    h, x = _inputs(torch, d.n_inputs, N_REUSE, 700 + len(name))
    ref = Reference(d, h)
    fused = sum(1 for j in d.joints if j.input_index >= 0) <= 7
    for k, form in enumerate(FORMS):
        wh, wd = _weights(torch, form, d.n_inputs, N_REUSE, 11 * k + len(name))
        for tau_h, tau_d in ((None, None), (h[3], x[3])):
            what = f"{name} {form} tau={'measured' if tau_h is not None else 'computed'}"
            _check(ch.regressorGram(*x[:3], tau_meas=tau_d, weights=wd), ref(wh, tau_h), what)
            flag, why = ch.gramKernelInfo()
            if fused:
                assert flag in (0, 1) and why.startswith("gram_fused_weighted_kernel, "), (what, flag, why)
            else:
                assert flag == 2 and why.startswith("general pipeline:"), (what, flag, why)


EXT_CASES = [("c6", 2), ("c6", 4), ("c7", 8), ("c7", 2), ("fold3_mix_tool", 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,xc", EXT_CASES)
def test_extended_model(name, xc, torch):
    """[Phi | Phi_c] with component sets that select XC = 2, 4, 8; C6, C7 and a chain with a prismatic joint; 100 003 samples; full planes
    and per-joint weights, computed and measured torques."""
    from rosdyn_b200.chain import Chain
    from test_instantiation_sweep import _set_components
    d = fixtures.by_name(name) if name in CHAINS else desc(name)
    ch = Chain(d)
    comps = components(d, xc)
    _set_components(ch, comps)
    n = 100_003
    h, x = _inputs(torch, d.n_inputs, n, 900 + xc)
    ref = Reference(d, h, comps)
    for form in ("plane", "joint"):
        wh, wd = _weights(torch, form, d.n_inputs, n, 13 + xc)
        for tau_h, tau_d in ((None, None), (h[3], x[3])):
            what = f"{name} XC={xc} {form} tau={'measured' if tau_h is not None else 'computed'}"
            _check(ch.regressorGramExt(*x[:3], tau_meas=tau_d, weights=wd), ref(wh, tau_h), what)
            flag, why = ch.gramKernelInfo()
            assert flag in (0, 1) and why.startswith("gram_fused_weighted_kernel, "), (what, flag, why)


def _paths():
    """(label, chain desc, component spec or None, environment): every kernel path the weighted entries take"""
    return [("c6 specialised", fixtures.by_name("c6"), None, {}), ("c7 precompiled", fixtures.by_name("c7"), None, {"RDB_GRAM_JIT": "0"}),
            ("generic generator", fixtures.by_name("random_a"), None, {}), ("folded", desc("fold5_mix_tool"), None, {}),
            ("general pipeline", desc("fold9_rev_plain"), None, {}), ("ext specialised", fixtures.by_name("c6"), 4, {}),
            ("ext precompiled", fixtures.by_name("c7"), 8, {"RDB_GRAM_JIT": "0"}), ("ext generic", fixtures.by_name("random_b"), 2, {}),
            ("ext general pipeline", desc("fold3_mix_tool"), "nine_columns", {}), ("unfed input", desc("k3_rev_unfed_input"), None, {})]


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(_paths())))
def test_unit_and_power_of_two_weights_are_exact(k, torch, monkeypatch):
    """w == 1 equals the unweighted entry bit for bit on every path (run-time specialised, RDB_GRAM_JIT=0, generic generator, folded chain,
    general pipeline, extended model); w == 4 and w == 1/4 give exactly 4x and 1/4x its outputs."""
    from rosdyn_b200.chain import Chain
    from test_instantiation_sweep import _set_components
    label, d, spec, env = _paths()[k]
    for key, v in env.items():
        monkeypatch.setenv(key, v)
    ch = Chain(d)
    if spec is not None:
        _set_components(ch, components(d, spec))
    ext = spec is not None
    n = 30_001
    _, x = _inputs(torch, d.n_inputs, n, 300 + k)
    call = ch.regressorGramExt if ext else ch.regressorGram
    for tau_d in (None, x[3]):
        base = call(*x[:3], tau_meas=tau_d)
        flag0 = ch.gramKernelInfo()[0]
        for form in ("scalar", "joint", "sample", "plane"):
            for c in (1.0, 4.0, 0.25):
                if form == "scalar":
                    w = torch.tensor(c, dtype=torch.float64, device="cuda")
                elif form == "joint":
                    w = torch.full((d.n_inputs,), c, dtype=torch.float64, device="cuda")
                elif form == "sample":
                    w = torch.full((n,), c, dtype=torch.float64, device="cuda")
                else:
                    w = torch.full((d.n_inputs, n + 3), c, dtype=torch.float64, device="cuda")[:, :n]
                out = call(*x[:3], tau_meas=tau_d, weights=w)
                assert ch.gramKernelInfo()[0] == flag0, f"{label}: the weighted call ran another kind of kernel"
                _equal(torch, out, tuple(v * c for v in base), f"{label} {form} w={c} tau={'measured' if tau_d is not None else 'computed'}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "random_c", "fold9_rev_plain"])
def test_one_hot_joint_weights(name, torch):
    """One-hot per-joint weights give G_r, b_r, tau_r^T tau_r: each matches the oracle, and their sum matches the unweighted call within
    1e-14 of its scale."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name) if name in CHAINS else desc(name)
    ch = Chain(d)
    n = 25_013
    h, x = _inputs(torch, d.n_inputs, n, 61)
    ref = Reference(d, h)
    G0, b0, t0 = (_np(v) for v in ch.regressorGram(*x[:3], tau_meas=x[3]))
    S = [np.zeros_like(G0), np.zeros_like(b0), 0.0]
    for r in range(d.n_inputs):
        wr = np.zeros(d.n_inputs)
        wr[r] = 1.0
        G, b, tt = (_np(v) for v in ch.regressorGram(*x[:3], tau_meas=x[3], weights=torch.tensor(wr, device="cuda")))
        assert_gram(G, b, tt, *ref(np.broadcast_to(wr[:, None], (d.n_inputs, n)), h[3]), f"{name}: joint {r}")
        S[0] += G
        S[1] += b
        S[2] += float(tt[0])
    assert np.max(np.abs(S[0] - G0)) <= 1e-14 * np.max(np.abs(G0)) * d.n_inputs
    assert np.max(np.abs(S[1] - b0)) <= 1e-14 * np.max(np.abs(b0)) * d.n_inputs
    assert abs(S[2] - float(t0[0])) <= 1e-14 * float(t0[0]) * d.n_inputs


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c7", "random_d"])
def test_zero_weight_window(name, torch):
    """A zero weight over [lo, hi) gives the unweighted normal equations of [0, lo) plus those of [hi, n)."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    n, lo, hi = 40_000, 7_001, 23_457
    _, x = _inputs(torch, d.n_inputs, n, 71)
    w = torch.ones(n, dtype=torch.float64, device="cuda")
    w[lo:hi] = 0.0
    Gw, bw, tw = (_np(v) for v in ch.regressorGram(*x[:3], tau_meas=x[3], weights=w))
    out = ch.regressorGram(*(v[:, :lo] for v in x[:3]), tau_meas=x[3][:, :lo])
    ch.regressorGram(*(v[:, hi:] for v in x[:3]), tau_meas=x[3][:, hi:], out=out)
    assert_gram(Gw, bw, tw, *(_np(v) for v in out[:2]), float(_np(out[2])[0]), f"{name}: masked window")


@pytest.mark.gpu
def test_unfed_input_measured_torque(torch):
    """Inputs no chain joint feeds: a zero regressor row, but their w tau^2 joins tau_sq (fused path and general pipeline)."""
    from rosdyn_b200.chain import Chain
    for name in ("k3_rev_unfed_input", "k9_rev_unfed_input"):
        d = desc(name)
        ch = Chain(d)
        n = 20_011
        h, x = _inputs(torch, d.n_inputs, n, 81)
        ref = Reference(d, h)
        for form in ("plane", "joint", "sample"):
            wh, wd = _weights(torch, form, d.n_inputs, n, 5)
            _check(ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd), ref(wh, h[3]), f"{name} {form}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7"])
def test_accuracy_at_scale(name, torch):
    """10^6 + 13 samples, full-plane weights, against the oracle's regressor contracted in float64 slices."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    n = 1_000_013
    h, x = _inputs(torch, d.n_inputs, n, 91, pad=0)
    wh, wd = _weights(torch, "plane", d.n_inputs, n, 17)
    ref = Reference(d, h)
    _check(ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd), ref(wh, h[3], step=65536), f"{name}: 10^6 samples")


def _solve_np(G, b, rel_tol=1e-10):
    """minimum-norm solution through the eigen-decomposition, eigenvalues <= rel_tol lambda_max discarded (rdb_normal_equations_solve)"""
    lam, V = np.linalg.eigh(G)
    keep = lam > rel_tol * lam.max()
    return V[:, keep] @ ((V[:, keep].T @ b) / lam[keep]), int(keep.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7"])
def test_wls_loop(name, torch):
    """Measured torques = model torque + seeded noise with per-joint sigma spread over 40x; OLS; sigma_j from the per-joint residuals of
    one-hot weighted Grams; WLS with w_j = 1 / sigma_j^2.  sigma_j and the WLS estimate match numpy's computation of the same quantities
    on the oracle regressor (same rank cut) to 1e-8 relative."""
    from rosdyn_b200.chain import Chain, solveNormalEquations
    d = fixtures.by_name(name)
    ch = Chain(d)
    n_in, n = d.n_inputs, 200_003
    h, x = _inputs(torch, n_in, n, 101)
    ref = Reference(d, h)
    sigma = np.geomspace(2.0, 0.05, n_in)  # 40x
    tau = ref.tau + np.random.RandomState(7).standard_normal((n_in, n)) * sigma[:, None]
    tau_d = torch.tensor(tau, device="cuda")
    # library
    G, b, tt = ch.regressorGram(*x[:3], tau_meas=tau_d)
    sol = solveNormalEquations(G, b, tt)
    pi = sol["parameters"]
    s_lib = np.zeros(n_in)
    for r in range(n_in):
        wr = torch.zeros(n_in, dtype=torch.float64, device="cuda")
        wr[r] = 1.0
        Gr, br, tr = (_np(v) for v in ch.regressorGram(*x[:3], tau_meas=tau_d, weights=wr))
        s_lib[r] = np.sqrt((float(tr[0]) - 2.0 * pi @ br + pi @ Gr @ pi) / n)
    Gw, bw, tw = ch.regressorGram(*x[:3], tau_meas=tau_d, weights=torch.tensor(1.0 / s_lib ** 2, device="cuda"))
    wls = solveNormalEquations(Gw, bw, tw)
    # numpy on the oracle regressor
    ones = np.ones((n_in, n))
    Gn, bn, _ = ref(ones, tau)
    pin, rank = _solve_np(Gn, bn)
    assert rank == sol["rank"], (rank, sol["rank"])
    X = ref.X
    resid = np.einsum("prs,p->rs", X, pin) - tau
    s_np = np.sqrt(np.sum(resid * resid, axis=1) / n)
    assert np.max(np.abs(s_lib / s_np - 1.0)) <= 1e-8, (s_lib, s_np)
    assert np.max(np.abs(s_np / sigma - 1.0)) < 0.05, (s_np, sigma)  # the loop recovers the noise levels
    Gwn, bwn, _ = ref(np.broadcast_to((1.0 / s_np ** 2)[:, None], (n_in, n)), tau)
    pwn, rank_w = _solve_np(Gwn, bwn)
    assert rank_w == wls["rank"]
    assert np.max(np.abs(wls["parameters"] - pwn)) <= 1e-8 * np.max(np.abs(pwn)), np.max(np.abs(wls["parameters"] - pwn))


@pytest.mark.gpu
def test_call_behaviour(torch):
    """Repeated launches are bit-reproducible; accumulate adds exactly; tau_sq = NULL is accepted; expanded views work; a call on a caller
    stream behind a bounded gate equals the solo call; host arrays are refused."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    n = 50_001
    h, x = _inputs(torch, d.n_inputs, n, 111)
    wh, wd = _weights(torch, "plane", d.n_inputs, n, 3)
    solo = ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd)
    _equal(torch, ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd), solo, "repeat")
    out = tuple(v.clone() for v in solo)
    ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd, out=out)
    _equal(torch, out, tuple(v + v for v in solo), "accumulate")
    # an expanded view: one weight per joint as a (n_in, n) view of stride (1, 0)
    wj = torch.linspace(0.5, 2.0, d.n_inputs, dtype=torch.float64, device="cuda")
    _equal(torch, ch.regressorGram(*x[:3], weights=wj[:, None].expand(d.n_inputs, n)), ch.regressorGram(*x[:3], weights=wj), "expanded view")
    # tau_sq = NULL through the C-ABI
    lib = _lib.load()
    P = 10 * d.n_joints
    G3 = torch.full((P, P), np.nan, dtype=torch.float64, device="cuda")
    b3 = torch.full((P,), np.nan, dtype=torch.float64, device="cuda")
    cw, _keep = ch._weights(True, n, wd)
    s = ch._samples(n, list(x[:3]) + [None])
    torch.cuda.synchronize()
    assert _c_call(lib, ch._h, ctypes.byref(s), ctypes.c_void_p(x[3].data_ptr()), ctypes.byref(cw), ctypes.c_void_p(G3.data_ptr()),
                   ctypes.c_void_p(b3.data_ptr()), None) == _lib.RDB_OK
    torch.cuda.synchronize()
    assert torch.equal(G3, solo[0]) and torch.equal(b3, solo[1])
    # caller stream behind a gate
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    done = torch.cuda.Event()
    with torch.cuda.stream(st):
        torch.cuda._sleep(200_000_000)  # a fraction of a second at the SM clock
        g = ch.regressorGram(*x[:3], tau_meas=x[3], weights=wd)
        done.record()
    time.sleep(0.02)
    assert not done.query(), "the gate did not hold the call"
    torch.cuda.synchronize()
    _equal(torch, g, solo, "caller stream")
    with pytest.raises(ValueError):
        ch.regressorGram(*(_np(v) for v in x[:3]), weights=np.ones(d.n_inputs))
    with pytest.raises(ValueError):
        ch.regressorGram(*x[:3], weights=torch.ones(d.n_inputs + 1, dtype=torch.float64, device="cuda"))


@pytest.mark.gpu
def test_facades(torch, tmp_path):
    """The C++ facade program runs; the Python methods return CUDA float64 tensors of the unweighted shapes."""
    exe = _build_cpp(str(tmp_path / "gram_weighted_check"))
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "weighted gram facade ok" in r.stdout, r.stdout + r.stderr
    from rosdyn_b200.chain import Chain
    ch = Chain(fixtures.by_name("c7"))
    _, x = _inputs(torch, 7, 500, 121)
    for t, shape in zip(ch.regressorGram(*x[:3], weights=torch.ones(500, dtype=torch.float64, device="cuda")), ((70, 70), (70,), (1,))):
        assert tuple(t.shape) == shape and t.is_cuda and t.dtype == torch.float64
