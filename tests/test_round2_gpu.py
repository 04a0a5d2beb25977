"""GPU parity, second tier (SURVEY.md section 8c acceptance): DIRECT oracle comparison of every entry point on 1e6 samples per chain with the
edge cases planted in the batch (q = 0, q = +-pi exactly, Dq = 0, DDq = 0, whole-circle angles), a zero-mass interior link, the fused normal
equations against the long-double oracle at 1e6 samples, the Eigen-record output layout, the NCCL group of the C-ABI, handles on other
devices and two host threads on one handle.  Tolerance: maxabs(x - ref) <= 1e-10 * max(maxabs(ref), 1) per output array."""
import concurrent.futures as cf
import copy
import ctypes
import math

import numpy as np
import pytest

from conftest import RTOL, assert_close, rel_err
from rosdyn_b200 import fixtures

pytestmark = pytest.mark.gpu

KIN = ("T_tool", "T_links", "jacobian", "twist", "dtwist", "dtwist_lin", "dtwist_nonlin", "ddtwist", "ddtwist_lin", "ddtwist_nonlin",
       "torque")
N_BIG = 1_000_000
CHUNK = 250_000


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _planted_inputs(n_in, n, seed):
    """U(-1,1) rates as the reference's tests draw them; angles over the whole circle; the first samples carry the edge cases."""
    from oracle.oracle import fill_uniform
    q, dq, ddq, dddq = (fill_uniform(n_in, n, seed, s) for s in range(4))
    q *= math.pi                      # whole circle
    q[:, 0] = 0.0
    q[:, 1] = math.pi                 # +pi exactly (the double nearest to pi)
    q[:, 2] = -math.pi
    q[:, 3] = np.where(np.arange(n_in) % 2 == 0, math.pi, -math.pi)
    dq[:, 4] = 0.0                    # Dq = 0
    ddq[:, 5] = 0.0
    dq[:, 6] = 0.0
    ddq[:, 6] = 0.0
    dddq[:, 6] = 0.0                  # a sample at rest
    q[:, 7] = math.pi / 2
    return q, dq, ddq, dddq


def _zero_mass_interior(name):
    """The chain with the inertial parameters of an interior moving link set to zero (mass, cog, inertia): its Phi block stays, pi_nom has zeros."""
    d = copy.deepcopy(fixtures.by_name(name))
    l = d.links[3]
    l.mass = 0.0
    l.cog = (0.0, 0.0, 0.0)
    l.inertia = (0.0,) * 6
    d.name = name + "_zero_mass_link3"
    return d


@pytest.mark.parametrize("name", ["c6", "c7", "c6_perturbed", "c7_perturbed", "random_a", "c6_zero_mass"])
def test_direct_oracle_comparison_1e6(name, torch):
    """Every output of every throughput entry point against the CPU restatement of primitives_impl.h on 1e6 samples (chunks of 250 k)."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = _zero_mass_interior("c6") if name == "c6_zero_mass" else fixtures.by_name(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in, P = d.n_inputs, 10 * d.n_joints
    worst = {}
    for c in range(N_BIG // CHUNK):
        hq, hdq, hddq, hdddq = _planted_inputs(n_in, CHUNK, 0x5EED0000 + 101 + c)
        q, dq, ddq, dddq = (torch.tensor(x, device="cuda") for x in (hq, hdq, hddq, hdddq))
        K = ch.kinematics(q, dq, ddq, dddq, want=KIN)
        R = oc.kinematics(hq, hdq, hddq, hdddq, nthreads=0)
        for k in KIN:
            worst[k] = max(worst.get(k, 0.0), rel_err(_np(K[k]), R[k]))
        del K, R
        rphi, rtau = oc.regressor_torque(hq, hdq, hddq, nthreads=0)
        phi, tau = ch.getRegressor(q, dq, ddq, with_torque=True)
        planes = _np(phi.transpose(0, 1).reshape(P * n_in, CHUNK))
        worst["regressor"] = max(worst.get("regressor", 0.0), rel_err(planes, rphi))
        Phi = planes.reshape(P, n_in, CHUNK)
        for j, jd in enumerate(d.joints):
            if jd.input_index >= 0:
                assert np.all(Phi[:10 * j, jd.input_index, :] == 0.0), "structural zeros must be exact"
        worst["torque(regressor pass)"] = max(worst.get("torque(regressor pass)", 0.0), rel_err(_np(tau), rtau))
        worst["torque"] = max(worst.get("torque", 0.0), rel_err(_np(ch.getJointTorque(q, dq, ddq)), rtau))
        del phi, planes, Phi, rphi
        M = ch.getJointInertia(q)
        worst["inertia"] = max(worst.get("inertia", 0.0), rel_err(_np(M.transpose(0, 1).reshape(n_in ** 2, CHUNK)), oc.inertia(hq, nthreads=0)))
        del M
    for k, e in worst.items():
        assert e <= RTOL, f"{name}:{k}: rel err {e:.3e} over {N_BIG} samples"


def _oracle_gram_parallel(oc, q, dq, ddq, tau=None, parts=16):
    """The long-double oracle over `parts` contiguous slices on host threads (the C call releases the GIL); partial sums added in order."""
    n = q.shape[1]
    cuts = [(k * n) // parts for k in range(parts + 1)]

    def one(k):
        s = slice(cuts[k], cuts[k + 1])
        return oc.gram(np.ascontiguousarray(q[:, s]), np.ascontiguousarray(dq[:, s]), np.ascontiguousarray(ddq[:, s]),
                       None if tau is None else np.ascontiguousarray(tau[:, s]))
    with cf.ThreadPoolExecutor(max_workers=parts) as ex:
        res = list(ex.map(one, range(parts)))
    G = sum(r[0] for r in res)
    b = sum(r[1] for r in res)
    return G, b, sum(r[2] for r in res)


@pytest.mark.parametrize("name", ["c6", "c7"])
def test_gram_against_long_double_oracle_1e6(name, torch):
    """SURVEY.md section 7 "summation order": 1e6-term fp64 sums in the GPU's tree order against sequential long-double accumulation."""
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch, oc = Chain(d), OracleChain(d)
    n = N_BIG + 13   # ragged
    hq, hdq, hddq = (fill_uniform(d.n_inputs, n, 0x5EED0000 + 202, s) for s in range(3))
    Gr, br, ttr = _oracle_gram_parallel(oc, hq, hdq, hddq)
    q, dq, ddq = (torch.tensor(x, device="cuda") for x in (hq, hdq, hddq))
    G, b, tt = ch.regressorGram(q, dq, ddq)
    G, b, tt = _np(G), _np(b), _np(tt)
    scale = np.max(np.abs(Gr))
    assert np.max(np.abs(G - Gr)) <= 1e-10 * scale, np.max(np.abs(G - Gr)) / scale
    assert np.max(np.abs(b - br)) <= 1e-10 * np.max(np.abs(br))
    assert abs(tt[0] - ttr) <= 1e-10 * ttr
    assert np.array_equal(G, G.T)
    # measured torques instead of the model's
    htau = fill_uniform(d.n_inputs, n, 0x5EED0000 + 203, 3) * 30.0
    Gr2, br2, ttr2 = _oracle_gram_parallel(oc, hq, hdq, hddq, htau)
    G2, b2, tt2 = ch.regressorGram(q, dq, ddq, tau_meas=torch.tensor(htau, device="cuda"))
    assert np.max(np.abs(_np(G2) - Gr2)) <= 1e-10 * scale
    assert np.max(np.abs(_np(b2) - br2)) <= 1e-10 * max(np.max(np.abs(br2)), 1.0)
    assert abs(_np(tt2)[0] - ttr2) <= 1e-10 * ttr2


@pytest.mark.parametrize("name", ["c6", "random_a", "random_c"])
def test_eigen_record_layout(name, torch):
    """RDB_LAYOUT_EIGEN: per-sample records laid out as the reference's Eigen objects (Affine3d 4x4 column-major images, VectorOfVector6d,
    column-major Jacobian / regressor / inertia) carry exactly the numbers of the SoA planes -- device entry and host entry."""
    from rosdyn_b200.chain import Chain, fill_uniform
    d = fixtures.by_name(name)
    ch = Chain(d)
    n_in, nL, P, n = d.n_inputs, d.n_links, 10 * d.n_joints, 3001
    q, dq, ddq, dddq = (fill_uniform(n_in, n, 0x5EED0000 + 303, s, device="cuda") for s in range(4))
    for host in (False, True):
        a = [(_np(x) if host else x) for x in (q, dq, ddq, dddq)]
        cv = (lambda t: t) if host else _np
        S = ch.kinematics(*a, want=KIN)
        E = ch.kinematics(*a, want=KIN, layout="eigen")
        T = cv(E["T_tool"])                                  # [n, 4, 4]
        assert np.array_equal(T[:, :3, :], np.moveaxis(cv(S["T_tool"]).reshape(3, 4, n), 2, 0))
        assert np.array_equal(T[:, 3, :], np.tile([0.0, 0.0, 0.0, 1.0], (n, 1)))
        Tl = cv(E["T_links"])                                # [n, nL, 4, 4]
        assert np.array_equal(Tl[:, :, :3, :], np.moveaxis(cv(S["T_links"]).reshape(nL, 3, 4, n), 3, 0))
        assert np.array_equal(Tl[:, :, 3, :], np.tile([0.0, 0.0, 0.0, 1.0], (n, nL, 1)))
        assert np.array_equal(cv(E["jacobian"]), np.transpose(cv(S["jacobian"]).reshape(n_in, 6, n), (2, 1, 0)))   # [n, 6, n_in]
        for k in KIN[3:-1]:
            assert np.array_equal(cv(E[k]), np.moveaxis(cv(S[k]).reshape(nL, 6, n), 2, 0)), k                    # [n, nL, 6]
        assert np.array_equal(cv(E["torque"]), cv(S["torque"]).T)
        # the raw record IS the Eigen memory image: Affine3d of sample 5 = 16 doubles column-major
        raw = cv(E["T_tool"]).transpose(0, 2, 1).reshape(n, 16)[5] if host else _np(E["T_tool"].transpose(-1, -2).reshape(n, 16))[5]
        assert np.array_equal(raw.reshape(4, 4, order="F"), T[5])
        Sd = ch.dynamics(a[0], a[1], a[2], want=("regressor", "torque", "inertia"))
        Ed = ch.dynamics(a[0], a[1], a[2], want=("regressor", "torque", "inertia"), layout="eigen")
        assert np.array_equal(cv(Ed["regressor"]), np.transpose(cv(Sd["regressor"]).reshape(P, n_in, n), (2, 1, 0)))   # [n, n_in, P]
        assert np.array_equal(cv(Ed["inertia"]), np.transpose(cv(Sd["inertia"]).reshape(n_in, n_in, n), (2, 1, 0)))
        assert np.array_equal(cv(Ed["torque"]), cv(Sd["torque"]).T)
        phi, tau = ch.getRegressor(a[0], a[1], a[2], with_torque=True)
        assert np.array_equal(cv(Sd["regressor"]), cv(phi).transpose(1, 0, 2).reshape(P * n_in, n))
        assert np.array_equal(cv(Sd["torque"]), cv(tau))


def test_group_single_device_matches_plain_entry(torch):
    """rdb_group_create(ndev = 1) / rdb_group_create_rank(nranks = 1): no collective, same numbers as rdb_regressor_gram_batch; accumulate adds."""
    from rosdyn_b200.chain import Chain, fill_uniform
    from rosdyn_b200.sharding import Group
    d = fixtures.by_name("c6")
    n = 100_003
    q, dq, ddq = (fill_uniform(6, n, 0x5EED0000 + 404, s, device="cuda") for s in range(3))
    G0, b0, t0 = Chain(d).regressorGram(q, dq, ddq)
    for grp in (Group(d, [0]), Group.from_torch_distributed(d, 0)):
        assert grp.ranks == 1
        (G, b, tt), = grp.gram([(q, dq, ddq)])
        torch.cuda.synchronize()
        assert torch.equal(G, G0) and torch.equal(b, b0) and torch.equal(tt, t0)
        (G2, b2, tt2), = grp.gram([(q, dq, ddq)], out=[(G.clone(), b.clone(), tt.clone())], accumulate=True)
        torch.cuda.synchronize()
        assert torch.equal(G2, 2 * G0) and torch.equal(b2, 2 * b0)


def test_group_all_reduce_over_nvlink(torch):
    """One process, every GPU of the box: rdb_regressor_gram_sharded (fused kernel per device + ONE ncclAllReduce of the packed partials) against
    the single-device normal equations of the whole batch, and against the host-sum entry rdb_regressor_gram_sharded_host."""
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    from rosdyn_b200.chain import Chain, fill_uniform
    from rosdyn_b200.sharding import Group, shard_range, sharded_gram_host
    d = fixtures.by_name("c7")
    n = 400_007
    q, dq, ddq = (fill_uniform(7, n, 0x5EED0000 + 505, s, device="cuda:0") for s in range(3))
    G0, b0, t0 = Chain(d, device=0).regressorGram(q, dq, ddq)
    grp = Group(d, list(range(ndev)))
    assert grp.ranks == ndev
    shards = []
    for r in range(ndev):
        lo, hi = shard_range(n, r, ndev)
        shards.append(tuple(x[:, lo:hi].to(f"cuda:{r}").contiguous() for x in (q, dq, ddq)))
    res = grp.gram(shards)
    for r in range(ndev):
        torch.cuda.synchronize(r)
    scale = float(G0.abs().max())
    for r, (G, b, tt) in enumerate(res):   # every device holds the full sum
        assert float((G.to("cuda:0") - G0).abs().max()) <= 1e-12 * scale, r
        assert float((b.to("cuda:0") - b0).abs().max()) <= 1e-12 * float(b0.abs().max())
        assert abs(float(tt[0]) - float(t0[0])) <= 1e-12 * float(t0[0])
    chains = [Chain(d, device=r) for r in range(ndev)]
    Gh, bh, th = sharded_gram_host(chains, _np(q), _np(dq), _np(ddq))
    assert np.max(np.abs(Gh - _np(res[0][0]))) <= 1e-12 * scale


def test_handle_keeps_its_device(torch):
    """A handle lives on the device it was created on whatever the caller's current device is (rdb_chain_create_on; ADVICE round 1)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d, device=1)
    torch.cuda.set_device(0)
    ch.setInputJointsName(ch.getActiveJointsName())          # re-upload from a thread whose current device is 0
    assert ch._lib.rdb_chain_device(ch._h) == 1
    hq, hdq, hddq = (fill_uniform(6, 5000, 7, s) for s in range(3))
    tau = ch.getJointTorque(hq, hdq, hddq)                   # host entry: staging must live on device 1
    G, b, tt = ch.regressorGram(hq, hdq, hddq)
    oc = OracleChain(d)
    _, rtau = oc.regressor_torque(hq, hdq, hddq, nthreads=0)
    assert_close(tau, rtau, "torque through a handle of device 1")
    Gr, _, _ = oc.gram(hq, hdq, hddq)
    assert np.max(np.abs(G - Gr)) <= 1e-10 * np.max(np.abs(Gr))
    assert torch.cuda.current_device() == 0                  # the caller's device is restored


def test_two_host_threads_on_one_handle(torch):
    """The *_host entries keep their staging pipeline in the handle: two threads on ONE handle are serialised by the per-handle lock."""
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch, oc = Chain(d), OracleChain(d)
    batches = [tuple(fill_uniform(6, 300_000 + 17 * k, 900 + k, s) for s in range(3)) for k in range(4)]
    refs = [oc.gram(*b) for b in batches[:2]]

    def work(k):
        if k < 2:
            return ch.regressorGram(*batches[k])
        return ch.getJointTorque(*batches[k])
    with cf.ThreadPoolExecutor(max_workers=4) as ex:
        res = list(ex.map(work, range(4))) + list(ex.map(work, range(4)))
    for k in (0, 1, 4, 5):
        G, b, tt = res[k]
        Gr, br, ttr = refs[k % 4]
        assert np.max(np.abs(G - Gr)) <= 1e-10 * np.max(np.abs(Gr))
        assert np.max(np.abs(b - br)) <= 1e-10 * np.max(np.abs(br))
    for k in (2, 3, 6, 7):
        _, rtau = oc.regressor_torque(*batches[k % 4], nthreads=0)
        assert_close(res[k], rtau, "torque from a shared handle")


def test_input_selection_drops_components_and_tau_shape_is_checked(torch):
    from rosdyn_b200.chain import Chain, fill_uniform
    d = fixtures.by_name("c6")
    ch = Chain(d)
    names = ch.getActiveJointsName()
    assert ch.setComponents([{"type": "friction1", "joint": names[5], "min_velocity": 0.01, "max_velocity": 3.0}]) == 2
    ch.setInputJointsName(names[:3])                # 3 inputs: the component's input index 5 no longer exists
    assert ch.getComponentColumns() == 0            # dropped, not left dangling (ADVICE round 1)
    q, dq, ddq = (fill_uniform(3, 1000, 5, s, device="cuda") for s in range(3))
    ch.regressorGram(q, dq, ddq)
    with pytest.raises(ValueError):                 # a shorter tau_meas would be read past its end
        ch.regressorGram(q, dq, ddq, tau_meas=q[:, :500])
    with pytest.raises(ValueError):
        ch.regressorGram(q, dq, ddq, tau_meas=q[:2])


@pytest.mark.parametrize("name", ["c6", "c7", "random_a"])
def test_gram_is_bit_reproducible(name, torch):
    """The producer / consumer handshake of the fused kernels (release / acquire counters; compute-sanitizer's racecheck does not model them
    and reports the slot stores against the fragment loads) leaves no timing dependence: repeated runs on the same inputs are bit-identical, for batches
    that end inside a group, a k-step and a slot."""
    from rosdyn_b200.chain import Chain, fill_uniform
    d = fixtures.by_name(name)
    ch = Chain(d)
    for n in (1_000_003, 37, 4096 + 5):
        q, dq, ddq = (fill_uniform(d.n_inputs, n, 0x5EED0000 + 606, s, device="cuda") for s in range(3))
        G0, b0, t0 = (x.clone() for x in ch.regressorGram(q, dq, ddq))
        for _ in range(4):
            G, b, tt = ch.regressorGram(q, dq, ddq)
            assert torch.equal(G, G0) and torch.equal(b, b0) and torch.equal(tt, t0)


def test_cpp_group_example(torch):
    """examples/group_check.cpp: rdb_group_create / rdb_regressor_gram_sharded from plain C++ on every GPU of the box (one GPU: no collective,
    same path) against the host-sum entry."""
    import os
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "build", "group_check")
    if not os.path.exists(exe):
        pytest.skip("build/group_check not built")
    r = subprocess.run([exe, str(torch.cuda.device_count()), "400003"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "group_check: ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("n", [1, 7, 64])
@pytest.mark.parametrize("layout", ["soa", "eigen"])
def test_small_host_calls_use_the_same_kernels(n, layout, torch):
    """Host-buffer calls small enough for the handle's mapped pinned buffer (the per-sample getters of the C++ facade) run the kernels in place on
    host memory; their results are bit-identical to the device entries on the same samples, and a large call afterwards is unaffected."""
    from oracle.oracle import fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6_perturbed")
    ch = Chain(d)
    hq, hdq, hddq, hdddq = (fill_uniform(d.n_inputs, n, 0x5EED0000 + 707, s) for s in range(4))
    dev = [torch.tensor(x, device="cuda") for x in (hq, hdq, hddq, hdddq)]
    want = ("T_tool", "T_links", "jacobian", "twist", "dtwist", "ddtwist", "torque")
    for _ in range(2):  # the second pass reuses the mapped buffer
        Kh = ch.kinematics(hq, hdq, hddq, hdddq, want=want, layout=layout)
        Kd = ch.kinematics(*dev, want=want, layout=layout)
        for k in want:
            assert isinstance(Kh[k], np.ndarray)
            assert np.array_equal(Kh[k], _np(Kd[k])), k
        Dh = ch.dynamics(hq, hdq, hddq, want=("regressor", "torque", "inertia"), layout=layout)
        Dd = ch.dynamics(*dev[:3], want=("regressor", "torque", "inertia"), layout=layout)
        for k in ("regressor", "torque", "inertia"):
            assert np.array_equal(Dh[k], _np(Dd[k])), k
    assert np.array_equal(ch.getJointTorque(hq, hdq, hddq), _np(ch.getJointTorque(*dev[:3])))
    big = 300_000
    bq, bdq, bddq = (fill_uniform(d.n_inputs, big, 0x5EED0000 + 708, s) for s in range(3))
    tb = ch.getJointTorque(bq, bdq, bddq)
    assert np.array_equal(tb[:, :1000], _np(ch.getJointTorque(*(torch.tensor(x[:, :1000].copy(), device="cuda") for x in (bq, bdq, bddq)))))


@pytest.mark.parametrize("layout", ["soa", "eigen"])
def test_pageable_host_calls_through_the_pinned_bounce_buffers(layout, torch):
    """numpy (pageable) arrays large enough for several chunks: the host entries gather / scatter them through the pinned mirror of the staging
    arena with host threads (HostPipe::bounce); results bit-identical to the device entries, for plane and record layouts, ragged last chunk."""
    from oracle.oracle import fill_uniform
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    n = 40_001
    hq, hdq, hddq, hdddq = (fill_uniform(d.n_inputs, n, 0x5EED0000 + 808, s) for s in range(4))
    dev = [torch.tensor(x, device="cuda") for x in (hq, hdq, hddq, hdddq)]
    want = ("T_tool", "T_links", "jacobian", "twist", "dtwist", "ddtwist", "torque")
    Kh = ch.kinematics(hq, hdq, hddq, hdddq, want=want, layout=layout)
    Kd = ch.kinematics(*dev, want=want, layout=layout)
    for k in want:
        assert np.array_equal(Kh[k], _np(Kd[k])), k
    Dh = ch.dynamics(hq, hdq, hddq, want=("regressor", "torque", "inertia"), layout=layout)
    Dd = ch.dynamics(*dev[:3], want=("regressor", "torque", "inertia"), layout=layout)
    for k in ("regressor", "torque", "inertia"):
        assert np.array_equal(Dh[k], _np(Dd[k])), k
    # a leading dimension larger than n on the host side (a view into a wider array)
    wide = np.zeros((d.n_inputs, n + 77))
    wide[:, :n] = hq
    assert np.array_equal(ch.getJointTorque(wide[:, :n], hdq, hddq), _np(ch.getJointTorque(*dev[:3])))
    Gh, bh, th = ch.regressorGram(hq, hdq, hddq)
    Gd, bd, td = ch.regressorGram(*dev[:3])
    assert np.max(np.abs(Gh - _np(Gd))) <= 1e-12 * np.max(np.abs(Gh)) and np.max(np.abs(bh - _np(bd))) <= 1e-12 * np.max(np.abs(bh))
