"""Canonical frames of the folded chain (csrc/fold.cpp): the frame of every revolute link is turned about its origin, x_old = Q x_new with
Q e_z = axis, so that the fused kernels hold the axis as the compile-time constant e_z.  CPU: Q itself, its parameter map, and through the
oracle the identity that makes the frame change invisible, Phi[:, block l] = Phi'[:, block l] T(Q_l^T, 0).  GPU: everything computed on the
folded chain (normal equations, extended model, torque, inertia, forward dynamics) against the oracle on chains with axis-aligned and oblique
axes and interior fixed joints."""
import copy
import ctypes

import numpy as np
import pytest

from conftest import RTOL, assert_close
from rosdyn_b200 import fixtures
from rosdyn_b200.descriptor import FIXED, REVOLUTE

ALIGNED = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
# all-revolute random chains (oblique axes, random origins) with interior fixed joints
RANDOM = {"rev_fixed_a": lambda: fixtures.random_chain(515, 7, p_prismatic=0.0, p_fixed=0.2),
          "rev_fixed_b": lambda: fixtures.random_chain(626, 8, p_prismatic=0.0, p_fixed=0.3)}


def _desc(name):
    return RANDOM[name]() if name in RANDOM else fixtures.by_name(name)


def _dp(x):
    return x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _Q(axis):
    from rosdyn_b200._lib import load
    a = np.ascontiguousarray(axis, dtype=np.float64)
    Q = np.zeros(9)
    assert load().rdb_fold_canonical_frame(_dp(a), _dp(Q)) == 0
    return Q.reshape(3, 3)


def _T(R, t):
    from rosdyn_b200._lib import load
    R, t, T = np.ascontiguousarray(R, dtype=np.float64), np.ascontiguousarray(t, dtype=np.float64), np.zeros((10, 10))
    assert load().rdb_fold_parameter_map(_dp(R), _dp(t), _dp(T)) == 0
    return T


def _unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v)


def test_random_chains_have_interior_fixed_joints():
    for name in RANDOM:
        types = [j.type for j in _desc(name).joints]
        assert REVOLUTE in types and all(t in (REVOLUTE, FIXED) for t in types)
        first, last = types.index(REVOLUTE), len(types) - 1 - types[::-1].index(REVOLUTE)
        assert FIXED in types[first:last], name


def test_aligned_axes_get_exact_signed_permutations():
    for ax in ALIGNED:
        Q = _Q(ax)
        assert np.array_equal(Q @ np.array([0.0, 0.0, 1.0]), np.array(ax, dtype=np.float64))
        assert set(np.abs(Q).ravel()) == {0.0, 1.0} and np.array_equal(np.abs(Q).sum(0), np.ones(3)) and np.array_equal(np.abs(Q).sum(1), np.ones(3))
        assert np.array_equal(Q @ Q.T, np.eye(3)) and round(np.linalg.det(Q)) == 1
    assert np.array_equal(_Q((0, 0, 1)), np.eye(3))


def test_oblique_axes_and_invalid_axes():
    from rosdyn_b200._lib import load
    rng = np.random.RandomState(5)
    for _ in range(200):
        ax = _unit(rng.normal(size=3))
        Q = _Q(ax)
        assert np.array_equal(Q[:, 2], ax)
        assert np.max(np.abs(Q @ Q.T - np.eye(3))) <= 1e-15 and abs(np.linalg.det(Q) - 1.0) <= 1e-15
    Q = np.zeros(9)
    for bad in ((0.0, 0.0, 0.0), (0.0, 0.0, 2.0)):
        assert load().rdb_fold_canonical_frame(_dp(np.array(bad)), _dp(Q)) != 0


def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def _params(m, c, Icog):
    Io = Icog + m * _skew(c) @ _skew(c).T
    return np.array([m, *(m * c), Io[0, 0], Io[0, 1], Io[0, 2], Io[1, 1], Io[1, 2], Io[2, 2]])


def test_parameter_map_of_the_frame_change():
    """T(Q^T, 0) refers a link's parameters to its canonical frame: rigid-body formulas, and exact for the aligned axes."""
    rng = np.random.RandomState(6)
    axes = [np.array(a, dtype=np.float64) for a in ALIGNED] + [_unit(rng.normal(size=3)) for _ in range(20)]
    for ax in axes:
        Q = _Q(ax)
        m, c = rng.uniform(0.1, 10), rng.normal(0, 0.2, 3)
        a = rng.normal(size=(3, 3))
        Icog = a @ a.T * 0.05 + np.eye(3) * 0.01
        pi_old, pi_new = _params(m, c, Icog), _params(m, Q.T @ c, Q.T @ Icog @ Q)
        T = _T(Q.T, np.zeros(3))
        assert np.max(np.abs(T @ pi_old - pi_new)) <= 1e-13 * np.max(np.abs(pi_new))
        if np.count_nonzero(ax) == 1:   # signed permutation: every entry of T is 0 or +-1, T pi is pi permuted with signs
            assert set(np.abs(T).ravel()) <= {0.0, 1.0} and np.array_equal(np.abs(T).sum(1), np.ones(10))


def _canonical(d):
    """The chain re-expressed with every revolute link in its canonical frame (x_old = Q_l x_new; other links keep theirs), and Q_l."""
    c = copy.deepcopy(d)
    Qs, Qp = [], np.eye(3)
    for jd, ld in zip(c.joints, c.links[1:]):
        Q = _Q(_unit(jd.axis)) if jd.type == REVOLUTE else np.eye(3)
        jd.rot = tuple((Qp.T @ np.array(jd.rot).reshape(3, 3) @ Q).ravel())
        jd.xyz = tuple(Qp.T @ np.array(jd.xyz))
        if jd.type == REVOLUTE:
            jd.axis = (0.0, 0.0, 1.0)
        ld.cog = tuple(Q.T @ np.array(ld.cog))
        ld.inertial_rot = tuple((Q.T @ np.array(ld.inertial_rot).reshape(3, 3)).ravel())
        Qs.append(Q)
        Qp = Q
    return c, Qs


@pytest.mark.parametrize("name", ["c6_perturbed", "c7", "rev_fixed_a", "rev_fixed_b"])
def test_regressor_block_in_the_canonical_frame_times_T(name):
    """Phi[:, block l] = Phi'[:, block l] T(Q_l^T, 0) on the oracle, Phi' the regressor of the chain in canonical frames; same torques."""
    from oracle.oracle import OracleChain
    d = _desc(name)
    dc, Qs = _canonical(d)
    rng = np.random.RandomState(7)
    q, dq, ddq = (rng.uniform(-np.pi, np.pi, (d.n_inputs, 64)) for _ in range(3))
    phi, tau = OracleChain(d).regressor_torque(q, dq, ddq)
    phic, tauc = OracleChain(dc).regressor_torque(q, dq, ddq)
    n, nj = phi.shape[1], d.n_joints
    phi, phic = phi.reshape(10 * nj, d.n_inputs, n), phic.reshape(10 * nj, d.n_inputs, n)
    for l, Q in enumerate(Qs):
        blk = slice(10 * l, 10 * l + 10)
        assert_close(np.einsum("cri,cp->pri", phic[blk], _T(Q.T, np.zeros(3))), phi[blk], f"{name}: link {l}", 1e-12)
    assert_close(tauc, tau, f"{name}: torque", 1e-12)


# ---------------------------------------------------------------------------------------------------------------------------------- GPU
GPU_CHAINS = ["c6", "c7", "c6_perturbed", "rev_fixed_a", "rev_fixed_b"]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_CHAINS)
def test_gram_against_oracle_and_bit_reproducible(name, torch):
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n = 40_000 + 7
    hq, hdq, hddq = (fill_uniform(d.n_inputs, n, 0x5EED0000 + 909, s) for s in range(3))
    hq = hq * np.pi
    Gr, br, ttr = oc.gram(hq, hdq, hddq)
    q, dq, ddq = (torch.tensor(x, device="cuda") for x in (hq, hdq, hddq))
    G, b, tt = (x.clone() for x in ch.regressorGram(q, dq, ddq))
    G2, b2, tt2 = ch.regressorGram(q, dq, ddq)
    assert torch.equal(G, G2) and torch.equal(b, b2) and torch.equal(tt, tt2)
    G, b, tt = _np(G), _np(b), _np(tt)
    assert np.max(np.abs(G - Gr)) <= 1e-10 * np.max(np.abs(Gr)), np.max(np.abs(G - Gr)) / np.max(np.abs(Gr))
    assert np.max(np.abs(b - br)) <= 1e-10 * np.max(np.abs(br))
    assert abs(tt[0] - ttr) <= 1e-10 * ttr
    assert np.array_equal(G, G.T)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7"])
def test_extended_gram_against_oracle(name, torch):
    from oracle import oracle
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in = d.n_inputs
    comps = [(1 + (k % 3), k % n_in, 0.05, 0.7) for k in range(n_in + 2)]
    tn = {1: "friction1", 2: "friction2", 3: "spring"}
    pc = ch.setComponents([{"type": tn[t], "joint": j, "min_velocity": lo, "max_velocity": hi} for t, j, lo, hi in comps])
    n = 3000
    rng = np.random.RandomState(8)
    q, dq, ddq = (rng.uniform(-1, 1, (n_in, n)) for _ in range(3))
    phi, tau_r = oc.regressor_torque(q, dq, ddq)
    ref_c = oracle.components_regressor(comps, n_in, q, dq)
    P = 10 * d.n_joints
    X = np.concatenate([phi.reshape(P, n_in, n), ref_c.reshape(pc, n_in, n)], axis=0)
    G_ref, b_ref = np.einsum("ari,bri->ab", X, X), np.einsum("ari,ri->a", X, tau_r)
    G, b, _ = ch.regressorGramExt(*(torch.tensor(x, device="cuda") for x in (q, dq, ddq)))
    assert_close(_np(G) / np.max(np.abs(G_ref)), G_ref / np.max(np.abs(G_ref)), "extended gram", 1e-11)
    assert_close(_np(b) / np.max(np.abs(b_ref)), b_ref / np.max(np.abs(b_ref)), "extended rhs", 1e-11)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_CHAINS)
def test_torque_inertia_forward_dynamics_on_the_folded_chain(name, torch):
    from oracle.oracle import OracleChain, fill_uniform
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in, n = d.n_inputs, 20_000
    hq, hdq, hddq = (fill_uniform(n_in, n, 0x5EED0000 + 919, s) for s in range(3))
    q, dq, ddq = (torch.tensor(x, device="cuda") for x in (hq, hdq, hddq))
    nt = OracleChain.max_threads()
    _, rtau = oc.regressor_torque(hq, hdq, hddq, nthreads=nt)
    assert_close(_np(ch.getJointTorque(q, dq, ddq)), rtau, f"{name}: torque", RTOL)
    M = oc.inertia(hq, nthreads=nt)
    assert_close(_np(ch.getJointInertia(q).transpose(0, 1).reshape(n_in ** 2, n)), M, f"{name}: inertia", RTOL)
    # forward dynamics: the torques of (q, Dq, DDq) solve back to DDq
    acc, info = ch.getJointAcceleration(q, dq, ch.getJointTorque(q, dq, ddq), with_info=True)
    assert int(info.abs().sum()) == 0
    assert_close(_np(acc), hddq, f"{name}: forward dynamics round trip", RTOL)
