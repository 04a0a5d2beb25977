"""Forward dynamics, ddq = M(q)^-1 (tau - h(q, Dq)): rdb_forward_dynamics_batch(_host), Chain.getJointAcceleration and the C++ facade.

The reference has no such function; its users compose getJointInertia (PI.h:1357-1379) and getJointTorqueNonLinearPart (PI.h:1285-1293) with
a dense solve.  That composition, evaluated by the CPU oracle, is what the GPU results are compared with (`oracle_fd`).
CPU: the composition itself round-trips (tau = torque(q, Dq, DDq) solves back to DDq), the entries refuse null arguments without a device,
and tests/cpp/forward_dynamics_check.cpp compiles and links.  GPU (-m gpu): parity on every test chain and on the generic (> 8 joint)
walker, input selections, singular M, sizes / strides / host paths bit for bit, 1e6 samples with planted edge cases, components, C++, Python.
Tolerance: maxabs(x - ref) <= 1e-10 * max(maxabs(ref), 1) per output array."""
import copy
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import CHAINS, ROOT, assert_close
from rosdyn_b200 import _lib, fixtures
from rosdyn_b200.descriptor import FIXED, LinkDesc

N = 20_000
GENERIC = {"generic9": lambda: fixtures.random_chain(909, 9, p_fixed=0.0), "generic11": lambda: fixtures.random_chain(777, 11, p_fixed=0.0)}


def _desc(name):
    return GENERIC[name]() if name in GENERIC else fixtures.by_name(name)


def oracle_fd(desc, q, dq, tau):
    """The reference's composition on the CPU oracle: M = getJointInertia(q), h = getJointTorque(q, Dq, 0), ddq = solve(M, tau - h) per
    sample over the inputs that a moving chain joint feeds (the others: ddq = 0).  dq / tau None = 0."""
    from oracle.oracle import OracleChain
    oc = OracleChain(desc)
    n_in, n = q.shape
    z = np.zeros_like(q)
    nt = OracleChain.max_threads()
    _, h = oc.regressor_torque(q, z if dq is None else dq, z, nthreads=nt)
    M = oc.inertia(q, nthreads=nt).reshape(n_in, n_in, n)            # plane col * n_in + row
    b = (z if tau is None else tau) - h
    fed = sorted(j.input_index for j in desc.joints if j.input_index >= 0 and j.type != FIXED)
    A = np.moveaxis(M, 2, 0).transpose(0, 2, 1)[:, fed][:, :, fed]    # [sample, row, col]
    out = np.zeros((n_in, n))
    if fed:
        out[fed] = np.linalg.solve(A, b[fed].T[:, :, None])[:, :, 0].T
    return out


def _inputs(n_in, n, seed):
    from oracle.oracle import fill_uniform
    return tuple(fill_uniform(n_in, n, seed, s) for s in range(3))


# ---------------------------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", CHAINS + list(GENERIC))
def test_oracle_composition_round_trip(name):
    """tau = getJointTorque(q, Dq, DDq) from the oracle; the composition the GPU tests compare with solves it back to DDq."""
    from oracle.oracle import OracleChain
    d = _desc(name)
    q, dq, ddq = _inputs(d.n_inputs, 4000, 0x5EED0000 + 901)
    _, tau = OracleChain(d).regressor_torque(q, dq, ddq)
    assert_close(oracle_fd(d, q, dq, tau), ddq, f"{name}: oracle composition round trip")


def test_null_arguments_without_a_device():
    lib = _lib.load()
    assert lib.rdb_forward_dynamics_batch(None, None, None, None, 0, None, None) == _lib.RDB_ERR_INVALID_ARG
    assert lib.rdb_forward_dynamics_batch_host(None, None, None, None, 0, None) == _lib.RDB_ERR_INVALID_ARG
    s = _lib.CSamples(1, 1, None, None, None, None)
    assert lib.rdb_forward_dynamics_batch(None, ctypes.byref(s), None, None, 1, None, None) == _lib.RDB_ERR_INVALID_ARG
    assert lib.rdb_forward_dynamics_batch_host(None, ctypes.byref(s), None, None, 1, None) == _lib.RDB_ERR_INVALID_ARG


def _build_cpp(out):
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "oracle", "shim"), "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "forward_dynamics_check.cpp"), "-o", out, "-L", os.path.join(ROOT, "rosdyn_b200"), "-lrosdyn_b200",
           "-Wl,-rpath," + os.path.join(ROOT, "rosdyn_b200")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return out


def test_cpp_facade_compiles_and_links(tmp_path):
    exe = _build_cpp(str(tmp_path / "fd_check"))
    if _lib.load().rdb_device_count() == 0:   # without a device the binary only reports that it linked
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


def _cuda(torch, *xs):
    return [None if x is None else torch.tensor(x, device="cuda") for x in xs]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CHAINS + list(GENERIC))
def test_parity(name, torch):
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch = Chain(d)
    q, dq, ddq = _inputs(d.n_inputs, N, 0x5EED0000 + 911)
    q_, dq_, ddq_ = _cuda(torch, q, dq, ddq)
    tau_ = ch.getJointTorque(q_, dq_, ddq_)
    acc, info = ch.getJointAcceleration(q_, dq_, tau_, with_info=True)
    assert info.dtype == torch.int32 and int(info.abs().sum()) == 0
    assert_close(_np(acc), ddq, f"{name}: round trip through the device torque")
    assert_close(_np(acc), oracle_fd(d, q, dq, _np(tau_)), f"{name}: against the oracle composition")


def _select(name, names_of):
    d = copy.deepcopy(fixtures.by_name(name))
    d.set_input_joints(names_of([j.name for j in d.joints if j.type != FIXED]))
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["permuted_partial", "unfed_input", "zero_gravity", "dq_null", "tau_null"])
def test_inputs(case, torch):
    from rosdyn_b200.chain import Chain
    if case == "permuted_partial":
        d = _select("c7_perturbed", lambda nm: [nm[4], nm[0], nm[2], nm[6]])
    elif case == "unfed_input":
        d = _select("c6", lambda nm: nm[:3] + ["not_a_joint"] + nm[4:])
    elif case == "zero_gravity":
        d = fixtures.by_name("c6_perturbed")
        d.gravity = (0.0, 0.0, 0.0)
    else:
        d = fixtures.by_name("random_b")
    ch = Chain(d)
    q, dq, ddq = _inputs(d.n_inputs, N, 0x5EED0000 + 913)
    if case == "dq_null":
        dq = None
    q_, dq_, ddq_ = _cuda(torch, q, dq, ddq)
    tau_ = ch.getJointTorque(q_, dq_, ddq_)
    tau = _np(tau_)
    if case == "tau_null":
        tau_, tau = None, None
    acc = _np(ch.getJointAcceleration(q_, dq_, tau_))
    assert_close(acc, oracle_fd(d, q, dq, tau), f"{case}: against the oracle composition")
    if case == "unfed_input":
        assert np.all(acc[3] == 0.0)
        ddq[3] = 0.0
    if case != "tau_null":
        assert_close(acc, ddq, f"{case}: round trip")


@pytest.mark.gpu
def test_singular_inertia_reports_info(torch):
    """A massless last link gives M(q) an exactly zero last row and column: every sample fails the Cholesky, ddq is NaN, nothing faults; a
    regular chain on the same inputs keeps info == 0."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    d.links[6] = LinkDesc("wrist_3_link")
    ch, ok = Chain(d), Chain(fixtures.by_name("c6"))
    q, dq, ddq = _inputs(6, 5000, 0x5EED0000 + 917)
    q_, dq_, ddq_ = _cuda(torch, q, dq, ddq)
    acc, info = ch.getJointAcceleration(q_, dq_, ddq_, with_info=True)
    assert bool((info == 1).all()) and bool(torch.isnan(acc).all())
    acc_h, info_h = ch.getJointAcceleration(q[:, :37], dq[:, :37], ddq[:, :37], with_info=True)   # the host twin's info plane
    assert np.all(info_h == 1) and np.all(np.isnan(acc_h))
    acc2, info2 = ok.getJointAcceleration(q_, dq_, ddq_, with_info=True)
    assert int(info2.abs().sum()) == 0 and bool(torch.isfinite(acc2).all())


def _raw(ch, torch, q, dq, tau, n, ld_in, ld_out):
    """rdb_forward_dynamics_batch on strided device planes; columns past n of the output keep their sentinel."""
    n_in = q.shape[0]
    def planes(x):
        t = torch.full((n_in, ld_in), 7.0, dtype=torch.float64, device="cuda")
        t[:, :n] = torch.tensor(x[:, :n], device="cuda")
        return t
    Q, DQ, T = planes(q), planes(dq), planes(tau)
    out = torch.full((n_in, ld_out), -3.0, dtype=torch.float64, device="cuda")
    info = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")
    s = _lib.CSamples(n, ld_in, Q.data_ptr(), DQ.data_ptr(), None, None)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(ch._lib.rdb_forward_dynamics_batch(ch._h, ctypes.byref(s), ctypes.c_void_p(T.data_ptr()), ctypes.c_void_p(out.data_ptr()), ld_out,
                                                  ctypes.c_void_p(info.data_ptr()), st))
    out, info = _np(out), _np(info)
    assert np.all(out[:, n:] == -3.0)
    return out[:, :n], info[:n]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 37, 4101])
def test_sizes_strides_and_host_paths(n, torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c7_perturbed")
    ch = Chain(d)
    q, dq, ddq = _inputs(7, max(n, 1), 0x5EED0000 + 919)
    tau = _np(ch.getJointTorque(*_cuda(torch, q, dq, ddq)))
    a, ia = _raw(ch, torch, q, dq, tau, n, n + 5, n + 11)
    b, ib = _raw(ch, torch, q, dq, tau, n, n + 5, n + 11)
    assert np.array_equal(a, b) and np.array_equal(ia, ib)                 # bit-identical across launches
    c, _ = _raw(ch, torch, q, dq, tau, n, max(n, 1), max(n, 1))
    assert np.array_equal(a, c)                                            # strides change nothing
    assert np.all(ia == 0)
    assert_close(a, ddq[:, :n], "round trip")
    # host twin: pageable numpy (mapped small-call path at these sizes), pinned buffers through the raw entry
    h, ih = ch.getJointAcceleration(q[:, :n], dq[:, :n], tau[:, :n], with_info=True)
    assert np.array_equal(h, a) and np.array_equal(ih, ia)
    pin = lambda x: torch.tensor(x[:, :n].copy()).pin_memory()           # noqa: E731
    Q, DQ, T = pin(q), pin(dq), pin(tau)
    out = torch.empty((7, max(n, 1)), dtype=torch.float64).pin_memory()
    info = torch.empty((max(n, 1),), dtype=torch.int32).pin_memory()
    s = _lib.CSamples(n, max(n, 1), Q.data_ptr(), DQ.data_ptr(), None, None)
    _lib.check(ch._lib.rdb_forward_dynamics_batch_host(ch._h, ctypes.byref(s), ctypes.c_void_p(T.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                       max(n, 1), ctypes.c_void_p(info.data_ptr())))
    assert np.array_equal(out.numpy()[:, :n], a) and np.array_equal(info.numpy()[:n], ia)


@pytest.mark.gpu
def test_large_host_calls_match_the_device_entry(torch):
    """Pageable (bounce buffers, two chunks) and pinned multi-chunk host calls are bit-identical to the device entry."""
    from oracle.oracle import fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6_perturbed")
    ch = Chain(d)
    n = 400_000
    q, dq, tau = (fill_uniform(6, n, 0x5EED0000 + 923, s) for s in range(3))
    tau *= 20.0
    dev, idev = ch.getJointAcceleration(*_cuda(torch, q, dq, tau), with_info=True)
    dev, idev = _np(dev), _np(idev)
    h, ih = ch.getJointAcceleration(q, dq, tau, with_info=True)
    assert np.array_equal(h, dev) and np.array_equal(ih, idev)
    p = [torch.tensor(x).pin_memory() for x in (q, dq, tau)]
    hp, ihp = ch.getJointAcceleration(*p, with_info=True)
    assert np.array_equal(hp, dev) and np.array_equal(ihp, idev)


def _planted(n_in, n, seed):
    """Angles over the whole circle, rates U(-1,1); the first samples carry q = 0, q = +-pi exactly, Dq = 0 and a sample at rest."""
    q, dq, ddq = _inputs(n_in, n, seed)
    q *= math.pi
    q[:, 0] = 0.0
    q[:, 1] = math.pi
    q[:, 2] = -math.pi
    q[:, 3] = np.where(np.arange(n_in) % 2 == 0, math.pi, -math.pi)
    dq[:, 4] = 0.0
    dq[:, 6] = 0.0
    ddq[:, 6] = 0.0
    q[:, 7] = math.pi / 2
    return q, dq, ddq


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7"])
def test_round_trip_1e6(name, torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    q, dq, ddq = _cuda(torch, *_planted(d.n_inputs, 1_000_000, 0x5EED0000 + 929))
    acc, info = ch.getJointAcceleration(q, dq, ch.getJointTorque(q, dq, ddq), with_info=True)
    assert int(info.abs().sum()) == 0
    assert_close(_np(acc), _np(ddq), f"{name}: 1e6 round trip")


@pytest.mark.gpu
def test_components_compose_by_subtraction(torch):
    """tau_eff = tau - Phi_c pi_c through rdb_components_torque_batch(-pi_c, accumulate = 1), then forward dynamics."""
    from oracle import oracle
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6_perturbed")
    ch = Chain(d)
    comps = [(1, 0, 0.05, 0.8), (2, 1, 0.1, 0.7), (3, 2, 0.0, 0.0), (1, 3, 0.01, 2.0), (2, 4, 0.02, 1.0), (3, 5, 0.0, 0.0)]
    tn = {1: "friction1", 2: "friction2", 3: "spring"}
    pc = ch.setComponents([{"type": tn[t], "joint": j, "min_velocity": lo, "max_velocity": hi} for t, j, lo, hi in comps])
    pi_c = np.linspace(0.5, 3.0, pc)
    q, dq, ddq = _inputs(6, N, 0x5EED0000 + 937)
    q_, dq_, ddq_ = _cuda(torch, q, dq, ddq)
    tau_ = ch.getJointTorque(q_, dq_, ddq_)
    tau = _np(tau_)
    eff = ch.getComponentsTorque(q_, dq_, -pi_c, out=tau_.clone())
    acc = _np(ch.getJointAcceleration(q_, dq_, eff))
    phi_c = oracle.components_regressor(comps, 6, q, dq).reshape(pc, 6, N)
    assert_close(acc, oracle_fd(d, q, dq, tau - np.einsum("cri,c->ri", phi_c, pi_c)), "friction / springs subtracted")


@pytest.mark.gpu
def test_cpp_facade_runs(tmp_path, torch):
    r = subprocess.run([_build_cpp(str(tmp_path / "fd_check"))], capture_output=True, text=True)
    assert r.returncode == 0 and "forward dynamics facade ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_python_interface(torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c7")
    ch = Chain(d)
    q, dq, ddq = _inputs(7, 64, 0x5EED0000 + 941)
    tau = _np(ch.getJointTorque(*_cuda(torch, q, dq, ddq)))
    dev = ch.getJointAcceleration(*_cuda(torch, q, dq, tau))
    assert dev.is_cuda and dev.shape == (7, 64)
    host = ch.getJointAcceleration(q, dq, tau)
    assert isinstance(host, np.ndarray) and np.array_equal(host, _np(dev))
    one = ch.getJointAcceleration(q[:, 5], dq[:, 5], tau[:, 5])
    assert one.shape == (7,) and np.array_equal(one, host[:, 5])
    one_i = ch.getJointAcceleration(q[:, 5], dq[:, 5], tau[:, 5], with_info=True)
    assert one_i[1] == 0 and np.array_equal(one_i[0], one)
    with pytest.raises(ValueError):
        ch.getJointAcceleration(q, dq, tau[:6])
    with pytest.raises(ValueError):
        ch.getJointAcceleration(q, dq, tau[:, :10])
    with pytest.raises(ValueError):
        ch.getJointAcceleration(*_cuda(torch, q, dq), tau)   # device q with a host tau
