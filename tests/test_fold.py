"""The parameter map behind the folded chain (csrc/fold.cpp): a body rigidly attached to link A through x_A = R x_B + t has, referred to
frame A, the inertial parameters T pi_B -- checked here against the rigid-body formulas evaluated independently in numpy, and through the
oracle: the regressor block of a link behind a fixed joint equals the block of its carrier link times T (which is what lets the fused
kernels skip such links)."""
import ctypes

import numpy as np
import pytest

from rosdyn_b200 import fixtures
from rosdyn_b200.descriptor import FIXED, rpy_to_rot


def _T(R, t):
    from rosdyn_b200._lib import load
    lib = load()
    dp = ctypes.POINTER(ctypes.c_double)
    R = np.ascontiguousarray(R, dtype=np.float64)
    t = np.ascontiguousarray(t, dtype=np.float64)
    T = np.zeros((10, 10))
    assert lib.rdb_fold_parameter_map(R.ctypes.data_as(dp), t.ctypes.data_as(dp), T.ctypes.data_as(dp)) == 0
    return T


def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def _params(m, c, Icog):
    Io = Icog + m * _skew(c) @ _skew(c).T        # inertia about the frame origin (spacevect_algebra.h:238)
    return np.array([m, *(m * c), Io[0, 0], Io[0, 1], Io[0, 2], Io[1, 1], Io[1, 2], Io[2, 2]])


def test_parameter_map_against_rigid_body_formulas():
    rng = np.random.RandomState(0)
    for _ in range(50):
        R = np.array(rpy_to_rot(*rng.uniform(-np.pi, np.pi, 3))).reshape(3, 3)
        t = rng.normal(0, 0.5, 3)
        m = rng.uniform(0.1, 10)
        c = rng.normal(0, 0.2, 3)
        a = rng.normal(size=(3, 3))
        Icog = a @ a.T * 0.05 + np.eye(3) * 0.01
        pi_B = _params(m, c, Icog)
        pi_A = _params(m, R @ c + t, R @ Icog @ R.T)       # the same body described in frame A
        T = _T(R, t)
        assert np.max(np.abs(T @ pi_B - pi_A)) <= 1e-13 * max(1.0, np.max(np.abs(pi_A)))
    assert np.array_equal(_T(np.eye(3), np.zeros(3)), np.eye(10))
    # composition: attaching C to B to A is attaching C to A with the composed transform
    R1 = np.array(rpy_to_rot(0.3, -0.7, 1.1)).reshape(3, 3); t1 = np.array([0.1, -0.2, 0.3])
    R2 = np.array(rpy_to_rot(-1.0, 0.2, 0.4)).reshape(3, 3); t2 = np.array([-0.05, 0.4, 0.0])
    assert np.max(np.abs(_T(R1, t1) @ _T(R2, t2) - _T(R1 @ R2, R1 @ t2 + t1))) <= 1e-13


@pytest.mark.parametrize("which", ["restatement", "reference"])
def test_regressor_block_behind_a_fixed_joint_is_the_carrier_block_times_T(which, golden):
    from oracle.oracle import OracleChain
    for name, carrier, attached in (("c6_perturbed", 5, 6),):
        d = fixtures.by_name(name)
        assert d.joints[attached].type == FIXED
        if which == "reference":   # the reference's own getRegressor, stored in tests/golden/ref_<chain>.npz (make_golden_ref.py)
            phi = golden("ref_" + name)["regressor"]
        else:
            rng = np.random.RandomState(2)
            q, dq, ddq = (rng.uniform(-1, 1, (d.n_inputs, 64)) for _ in range(3))
            phi, _ = OracleChain(d).regressor_torque(q, dq, ddq)
        n = phi.shape[1]
        phi = phi.reshape(10 * d.n_joints, d.n_inputs, n)                   # [col][row][sample]
        j = d.joints[attached]
        T = _T(np.array(j.rot).reshape(3, 3), np.array(j.xyz))
        A = phi[10 * carrier:10 * carrier + 10]                              # block of the carrier link
        B = phi[10 * attached:10 * attached + 10]                            # block of the link behind the fixed joint
        assert np.max(np.abs(np.einsum("cri,cp->pri", A, T) - B)) <= 1e-12 * np.max(np.abs(B))
