"""CPU-only: the restatement oracle against the REFERENCE ITSELF.

* tests/golden/ref_<chain>.npz were produced by the reference's own rosdyn::Chain (its headers compiled where they lie under
  /root/reference against the stand-in third-party headers of oracle/shim/; generator tests/golden/make_golden_ref.py).
* when oracle/_ref/librosdyn_ref.so is present (built by __graft_entry__.build() when the reference sources are available) the oracle is
  also compared live on seeded batches, including permuted / partial input-joint lists and multi-threaded clones (Chain::clone)."""
import numpy as np
import pytest

from conftest import CHAINS, assert_close
from oracle import oracle
from oracle.oracle import OracleChain, fill_uniform
from rosdyn_b200 import fixtures

KIN = ("T_links", "jacobian", "twist", "dtwist", "dtwist_lin", "dtwist_nonlin", "ddtwist", "ddtwist_lin", "ddtwist_nonlin", "torque")
TOL = 1e-12  # both sides evaluate the same formulas in fp64; only the rounding order of the dense products differs


@pytest.mark.parametrize("name", CHAINS)
@pytest.mark.parametrize("fast", [False, True])
def test_oracle_matches_reference_outputs(name, fast, golden):
    g = golden("ref_" + name)
    oc = OracleChain(fixtures.by_name(name), fast=fast)
    tol = 1e-10 if fast else TOL  # the -Ofast build reassociates
    K = oc.kinematics(g["q"], g["dq"], g["ddq"], g["dddq"])
    for k in KIN:
        assert_close(K[k], g[k], f"{name}:{k}", tol)
    phi, tau = oc.regressor_torque(g["q"], g["dq"], g["ddq"])
    assert_close(phi, g["regressor"], f"{name}:regressor", tol)
    assert_close(tau, g["torque"], f"{name}:torque", tol)
    assert_close(oc.kinematics(g["q"], g["dq"], None, want=("torque",))["torque"], g["torque_nonlin"], f"{name}:torque_nonlin", tol)
    assert_close(oc.inertia(g["q"]), g["inertia"], f"{name}:inertia", tol)
    assert_close(oc.nominal_parameters(), g["nominal"], f"{name}:nominal", tol)
    pt, tt = oc.regressor_torque(g["q"], g["dq"], g["ddq"], nthreads=2)
    assert_close(pt, g["regressor"], f"{name}:regressor, 2 threads", tol)
    assert_close(tt, g["torque"], f"{name}:torque, 2 threads", tol)
    # normal equations: the sums oracle/_ref's oracle_regressor_gram forms from the reference's getRegressor / getJointTorque
    d = fixtures.by_name(name)
    Y = g["regressor"].reshape(10 * d.n_joints, d.n_inputs, -1)              # [col][row][sample]
    Gr, br, tr = np.einsum("crs,drs->cd", Y, Y), np.einsum("crs,rs->c", Y, g["torque"]), float(np.sum(g["torque"] ** 2))
    G, b, t2 = oc.gram(g["q"], g["dq"], g["ddq"])
    assert_close(G / np.max(np.abs(Gr)), Gr / np.max(np.abs(Gr)), f"{name}:gram", tol)
    assert_close(b / np.max(np.abs(br)), br / np.max(np.abs(br)), f"{name}:rhs", tol)
    assert abs(t2 - tr) <= tol * tr
    # structural zeros (row of chain joint j, column blocks of the links before it) are exact zeros on both sides
    for j, jd in enumerate(d.joints):
        if jd.input_index >= 0:
            rows = [c * d.n_inputs + jd.input_index for c in range(10 * j)]
            assert np.all(g["regressor"][rows] == 0.0) and np.all(phi[rows] == 0.0)


needs_ref = pytest.mark.skipif(not (oracle.have_ref() or oracle.build_ref()), reason="oracle/_ref/librosdyn_ref.so not built (needs /root/reference)")


@needs_ref
@pytest.mark.parametrize("name", CHAINS)
def test_oracle_matches_reference_live(name):
    d = fixtures.by_name(name)
    oc, rc = OracleChain(d), OracleChain(d, fast="ref")
    assert oracle.lib("ref").lib.oracle_kind() == b"reference"
    n = 400
    q, dq, ddq, dddq = (fill_uniform(d.n_inputs, n, 0xABC0 + len(name), s) for s in range(4))
    q *= 3.0
    a, b = oc.kinematics(q, dq, ddq, dddq), rc.kinematics(q, dq, ddq, dddq, nthreads=2)
    for k in a:
        assert_close(a[k], b[k], f"{name}:{k}", TOL)
    pa, ta = oc.regressor_torque(q, dq, ddq)
    pb, tb = rc.regressor_torque(q, dq, ddq, nthreads=2)
    assert_close(pa, pb, f"{name}:regressor", TOL)
    assert_close(ta, tb, f"{name}:torque", TOL)
    assert_close(oc.inertia(q), rc.inertia(q), f"{name}:inertia", TOL)
    Ga, ba, ta2 = oc.gram(q, dq, ddq)
    Gb, bb, tb2 = rc.gram(q, dq, ddq)
    assert_close(Ga / np.max(np.abs(Gb)), Gb / np.max(np.abs(Gb)), f"{name}:gram", TOL)
    assert_close(ba / np.max(np.abs(bb)), bb / np.max(np.abs(bb)), f"{name}:rhs", TOL)
    assert abs(ta2 - tb2) <= TOL * abs(tb2)


@needs_ref
def test_reference_input_joint_selection():
    """Chain::setInputJointsName (primitives_impl.h:705-742) with a permuted subset, and an input that names no chain joint."""
    names = [j.name for j in fixtures.by_name("c6").joints if j.type != 0]
    d = fixtures.by_name("c6")
    assert d.set_input_joints([names[i] for i in (3, 0, 5, 1)])
    oc, rc = OracleChain(d), OracleChain(d, fast="ref")
    q, dq, ddq = (fill_uniform(4, 50, 9, s) for s in range(3))
    for k, v in oc.kinematics(q, dq, ddq, want=("T_tool", "jacobian", "torque")).items():
        assert_close(v, rc.kinematics(q, dq, ddq, want=(k,))[k], k, TOL)
    assert_close(oc.regressor_torque(q, dq, ddq)[0], rc.regressor_torque(q, dq, ddq)[0], "regressor", TOL)
    assert_close(oc.inertia(q), rc.inertia(q), "inertia", TOL)
    d2 = fixtures.by_name("c6")
    d2.set_input_joints(names[:3] + ["not_a_joint"] + names[4:])   # input 3 feeds nothing
    o2, r2 = OracleChain(d2), OracleChain(d2, fast="ref")
    q, dq, ddq = (fill_uniform(6, 50, 10, s) for s in range(3))
    assert_close(o2.regressor_torque(q, dq, ddq)[0], r2.regressor_torque(q, dq, ddq)[0], "regressor with an unlisted input", TOL)
    assert_close(o2.kinematics(q, dq, ddq, want=("torque",))["torque"], r2.kinematics(q, dq, ddq, want=("torque",))["torque"], "torque", TOL)


def test_reference_ur10_known_answer(golden):
    """The reference's tool pose of C6 at the zero pose (sample 0 of tests/golden/ref_c6.npz has q = 0; the tool is the last link), and the
    restatement's at the same pose."""
    g = golden("ref_c6")
    assert np.all(g["q"][:, 0] == 0.0)
    T = g["T_links"][-12:, 0].reshape(3, 4)
    np.testing.assert_allclose(T[:, 3], [1.1843, 0.256141, 0.0116], atol=1e-12)
    T = OracleChain(fixtures.by_name("c6")).kinematics(np.zeros((6, 1)), want=("T_tool",))["T_tool"][:, 0].reshape(3, 4)
    np.testing.assert_allclose(T[:, 3], [1.1843, 0.256141, 0.0116], atol=1e-12)
