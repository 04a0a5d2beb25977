"""The entries on caller streams (include/rosdyn_b200.h, "stream" conventions).

torch's streams are non-blocking: the legacy default stream does not order them, so a call made under `with torch.cuda.stream(s)` runs
concurrently with everything on other streams unless the library orders it.  What is checked here:

1. every device entry is ordered on the caller's stream: behind a gate on a fresh stream the inputs are copied in (they hold NaN before),
   the outputs filled, then the entry called -- the result equals the same call run alone on the default stream, bit for bit;
2. two Gram calls of one handle on two streams (and a host Gram call while a device one is in flight) both return what they return alone:
   they share the handle's workspace (per-CTA partials, the folded chain's reduced normal equations, the extended model's blocks, the
   general pipeline's materialised regressor, the group's packed buffer);
3. the Gram calls of one handle are ordered across streams: a call on a second stream does not finish while the first one waits behind a
   gate, and the host Gram entry returns only after it;
4. a model change (setInputJointsName) waits for the calls already queued: they complete on the old input order, calls issued after it see
   the new one;
5. the entries that only read the handle run concurrently on distinct streams of one handle.

The gate is torch.cuda._sleep: a bounded spin of one thread on the SM clock, measured once per module.  Every entry is deterministic per
sample and per launch, so results are compared bit for bit; the solo results of the configurations no other test covers (C6 with friction on
every joint, C6 with a component set the one-pass kernel refuses) are also checked against the oracle.  Every tensor and handle is held until
after the final synchronisation."""
import copy
import time

import numpy as np
import pytest

from rosdyn_b200 import fixtures
from test_instantiation_sweep import KIN, _ext_reference, _oracle_gram, _set_components, assert_gram, desc

pytestmark = pytest.mark.gpu

NAN = float("nan")


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def gate(torch):
    """gate(seconds): torch.cuda._sleep on the current stream for about `seconds`, at the SM clock measured here with CUDA events"""
    torch.cuda._sleep(1000)
    cycles = 50_000_000
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    torch.cuda._sleep(cycles)
    b.record()
    b.synchronize()
    hz = cycles / (a.elapsed_time(b) * 1e-3)
    assert 1e8 < hz < 1e10, hz

    def g(seconds):
        torch.cuda._sleep(int(hz * seconds))
    return g


def _np(t):
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)


def _same(x, ref, what):
    x, ref = _np(x), _np(ref)
    assert x.shape == ref.shape and x.dtype == ref.dtype, (what, x.shape, ref.shape)
    eq = np.array_equal(x, ref, equal_nan=True) if x.dtype.kind == "f" else np.array_equal(x, ref)
    if not eq:
        bad = ~((x == ref) | (np.isnan(x) & np.isnan(ref))) if x.dtype.kind == "f" else x != ref
        pytest.fail(f"{what}: {int(bad.sum())} of {x.size} values differ from the solo run, e.g. {x[bad].ravel()[:3]} vs {ref[bad].ravel()[:3]}")


def _uniform(torch, n_in, n, seed):
    rng = np.random.RandomState(seed)
    h = [rng.uniform(-np.pi, np.pi, (n_in, n)), rng.uniform(-2, 2, (n_in, n)), rng.uniform(-5, 5, (n_in, n))]
    return h, [torch.tensor(x, device="cuda") for x in h]


def _big(n_in, n, seed):
    """a large device batch without a host round trip: q, Dq, DDq, and measured torques"""
    from rosdyn_b200.chain import fill_uniform
    return [fill_uniform(n_in, n, seed, s, device="cuda") for s in range(3)] + [fill_uniform(n_in, n, seed + 1, 3, device="cuda") * 30.0]


C6_COMPONENTS = [(1, 0, 0.05, 0.7), (3, 1, 0.0, 0.0), (2, 5, 0.1, 0.9)]   # friction1, spring, friction2: the one-pass extended kernel


# --------------------------------------------------------------------------------------------------- 1. ordered on the caller's stream
def _entry(torch, name, monkeypatch):
    """(real inputs [device tensors], call(xs) -> outputs, kernel info of the last Gram call or None) of one device entry"""
    from rosdyn_b200.chain import Chain, fill_uniform
    from rosdyn_b200.sharding import Group
    n = 4099
    chain = "unf9_rev" if name.endswith("_generic") else ("fold9_rev_plain" if name == "gram_general" else
                                                          ("k3_rev_unfed_input" if name == "gram_unfed_measured_tau" else None))
    d = desc(chain) if chain else fixtures.by_name("c6")
    ch = Chain(d)
    n_in, nL = d.n_inputs, d.n_joints + 1
    _, x = _uniform(torch, n_in, n, 11)
    if name.startswith("kinematics"):
        layout = "eigen" if "eigen" in name else "soa"
        x = x + [torch.tensor(np.random.RandomState(12).uniform(-9, 9, (n_in, n)), device="cuda")]
        return x, lambda xs: tuple(ch.kinematics(*xs, want=KIN, layout=layout).values()), None
    if name.startswith("dynamics"):
        layout = "eigen" if "eigen" in name else "soa"
        return x, lambda xs: tuple(ch.dynamics(*xs, want=("regressor", "torque", "inertia"), layout=layout).values()), None
    if name == "torque":
        return x, lambda xs: (ch.getJointTorque(*xs),), None
    if name == "regressor":
        return x, lambda xs: ch.getRegressor(*xs, with_torque=True), None
    if name == "inertia":
        return x[:1], lambda xs: (ch.getJointInertia(xs[0]),), None
    if name == "forward_dynamics":
        return x, lambda xs: ch.getJointAcceleration(xs[0], xs[1], xs[2] * 20.0, with_info=True), None
    if name == "wrench":
        ext = torch.tensor(np.random.RandomState(13).normal(size=(nL, 6, n)) * 10.0, device="cuda")
        return x + [ext], lambda xs: ch.getWrench(*xs[:3], xs[3], with_torque=True), None
    if name == "jacobian_link":
        return x[:1], lambda xs: (ch.getJacobianLink(xs[0], ch.getLinksName()[3]),), None
    if name == "local_ik":
        goal = torch.tensor(np.random.RandomState(14).uniform(-1, 1, (n_in, n)), device="cuda")
        target = ch.kinematics(goal, want=("T_tool",))["T_tool"].clone()
        seed = goal + torch.tensor(np.random.RandomState(15).uniform(-0.3, 0.3, (n_in, n)), device="cuda")
        lim = np.full(n_in, 2.5)
        return [target, seed], lambda xs: ch.computeLocalIk(xs[0], xs[1], -lim, lim, toll=1e-9, max_iter=30), None
    if name.startswith("components"):
        _set_components(ch, C6_COMPONENTS)
        if name == "components_regressor":
            return x[:2], lambda xs: (ch.getComponentsRegressor(*xs),), None
        prm = np.random.RandomState(16).uniform(-3, 3, ch.getComponentColumns())
        base = torch.tensor(np.random.RandomState(17).uniform(-9, 9, (n_in, n)), device="cuda")
        # the accumulate base is written on the stream of the call, behind the gate
        return x[:2], lambda xs: (ch.getComponentsTorque(*xs, prm, out=base.clone()),), None
    if name.startswith("gram"):
        ext = name == "gram_extended"
        if ext:
            _set_components(ch, C6_COMPONENTS)
        if name == "gram_fused_precompiled":
            monkeypatch.setenv("RDB_GRAM_JIT", "0")
        if name == "gram_general":
            x = _uniform(torch, n_in, 20011, 18)[1]
        P = 10 * d.n_joints + ch.getComponentColumns() * ext
        tau = [x[0] * 30.0] if name == "gram_unfed_measured_tau" else []
        gram = ch.regressorGramExt if ext else ch.regressorGram
        flag = {"gram_fused_jit": 1, "gram_fused_precompiled": 0, "gram_general": 2}.get(name)
        def call(xs):
            out = (torch.zeros((P, P), dtype=torch.float64, device="cuda"), torch.zeros(P, dtype=torch.float64, device="cuda"),
                   torch.zeros(1, dtype=torch.float64, device="cuda"))
            return gram(*xs[:3], tau_meas=xs[3] if tau else None, out=out)
        return x + tau, call, (lambda: ch.gramKernelInfo()) if flag is not None else None
    if name == "group_gram":
        grp = Group(d, [0])
        return x, lambda xs: grp.gram([tuple(xs)], streams=[torch.cuda.current_stream().cuda_stream])[0], None
    if name == "fill_uniform":
        def call(xs):
            # the block the result lands in holds NaN, written on this stream behind the gate
            t = torch.full((6, n), NAN, dtype=torch.float64, device="cuda")
            p = t.data_ptr()
            del t
            r = fill_uniform(6, n, 0x5EED, 1, device="cuda")
            assert r.data_ptr() == p, "the caching allocator did not hand back the NaN block"
            return (r,)
        return [], call, None
    raise KeyError(name)


ENTRIES = ["kinematics_soa", "kinematics_eigen", "kinematics_soa_generic", "kinematics_eigen_generic", "dynamics_soa", "dynamics_eigen",
           "torque", "regressor", "inertia", "forward_dynamics", "wrench", "jacobian_link", "local_ik", "components_regressor",
           "components_torque_accumulate", "gram_fused_jit", "gram_fused_precompiled", "gram_extended", "gram_general",
           "gram_unfed_measured_tau", "group_gram", "fill_uniform"]


@pytest.mark.parametrize("name", ENTRIES)
def test_device_entry_is_ordered_on_the_callers_stream(name, torch, gate, monkeypatch):
    real, call, check = _entry(torch, name, monkeypatch)
    torch.cuda.synchronize()
    solo = [_np(v) for v in call(real)]
    torch.cuda.synchronize()
    xs = [torch.full_like(r, NAN) for r in real]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        gate(0.2)
        for x, r in zip(xs, real):
            x.copy_(r)
        out = call(xs)
    torch.cuda.synchronize()
    assert len(out) == len(solo)
    for k, (u, v) in enumerate(zip(out, solo)):
        _same(u, v, f"{name}: output {k}")
    assert any(np.isfinite(v).any() for v in solo if v.dtype.kind == "f")
    if check is not None:  # the stream run took the kernel the case is named after
        flag = {"gram_fused_jit": 1, "gram_fused_precompiled": 0, "gram_general": 2}[name]
        assert check()[0] == flag, check()


# ----------------------------------------------------------------------------------------------- 2. two Gram calls on two streams
# case: (chain, components, samples of A, samples of B, measured torques for B)
GRAM_CASES = {
    "c6_fused_folded": ("c6", None, 16_000_000, 300_007, False),
    "c7_fused": ("c7", None, 16_000_000, 250_013, True),
    "c6_friction_every_joint": ("c6", "friction", 8_000_000, 50_021, True),
    "k9_general_pipeline": ("fold9_rev_plain", None, 2_000_000, 60_017, False),
    "c6_refused_components": ("c6", "nine_columns", 1_000_000, 30_011, True),
    "k3_unfed_input_measured_tau": ("k3_rev_unfed_input", None, 16_000_000, 300_007, True),
}


def _gram_case(name):
    from rosdyn_b200.chain import Chain
    chain, spec, na, nb, tb = GRAM_CASES[name]
    d = fixtures.by_name(chain) if chain in ("c6", "c7") else desc(chain)
    ch = Chain(d)
    comps = None
    if spec == "friction":
        comps = [(1, i, 0.05, 0.7) for i in range(d.n_inputs)]
    elif spec == "nine_columns":
        comps = [(2, 0, 0.05, 0.7)] * 3
    if comps:
        _set_components(ch, comps)
    # the unfed-input scratch word is used with measured torques only: A carries them there too
    ta = name.startswith("k3_unfed")
    return d, ch, comps, na, nb, ta, tb


def _dev_gram(ch, comps, x, tau):
    return (ch.regressorGramExt if comps else ch.regressorGram)(*x, tau_meas=tau)


@pytest.mark.parametrize("b_on", ["device", "host"])
@pytest.mark.parametrize("name", list(GRAM_CASES))
def test_two_gram_calls_on_two_streams_of_one_handle(name, b_on, torch):
    from oracle.oracle import OracleChain
    d, ch, comps, na, nb, ta, tb = _gram_case(name)
    n_in = d.n_inputs
    A = _big(n_in, na, 0x5EED0000 + 21)
    hB, B = _uniform(torch, n_in, nb, 22)
    htB = np.random.RandomState(23).uniform(-50, 50, (n_in, nb)) if tb else None
    tB = torch.tensor(htB, device="cuda") if tb else None
    a_tau = A[3] if ta else None
    torch.cuda.synchronize()
    solo_a = [_np(v) for v in _dev_gram(ch, comps, A[:3], a_tau)]
    if b_on == "device":
        solo_b = [_np(v) for v in _dev_gram(ch, comps, B, tB)]
        if comps:   # the component sets no other test runs on C6
            assert_gram(*solo_b, *_ext_reference(d, OracleChain(d), hB, comps, htB), f"{name}: solo B against the oracle")
        else:
            assert_gram(*solo_b, *_oracle_gram(OracleChain(d), hB, htB), f"{name}: solo B against the oracle")
    else:
        solo_b = [v.copy() for v in ch.regressorGram(*hB, tau_meas=htB)]   # the host entry: rigid-body normal equations
    torch.cuda.synchronize()
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        ra = _dev_gram(ch, comps, A[:3], a_tau)
    if b_on == "device":
        with torch.cuda.stream(sb):
            rb = _dev_gram(ch, comps, B, tB)
    else:
        rb = ch.regressorGram(*hB, tau_meas=htB)
    torch.cuda.synchronize()
    for k, (u, v) in enumerate(zip(ra, solo_a)):
        _same(u, v, f"{name}: A ({na} samples on stream A), output {k}")
    for k, (u, v) in enumerate(zip(rb, solo_b)):
        _same(u, v, f"{name}: B ({nb} samples, {b_on} entry), output {k}")


def test_group_gram_on_two_streams(torch):
    from rosdyn_b200.sharding import Group
    d = fixtures.by_name("c6")
    grp = Group(d, [0])
    A = _big(6, 16_000_000, 0x5EED0000 + 31)[:3]
    _, B = _uniform(torch, 6, 300_007, 32)
    torch.cuda.synchronize()
    solo_a = [_np(v) for v in grp.gram([tuple(A)])[0]]
    solo_b = [_np(v) for v in grp.gram([tuple(B)])[0]]
    torch.cuda.synchronize()
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    ra = grp.gram([tuple(A)], streams=[sa.cuda_stream])[0]
    rb = grp.gram([tuple(B)], streams=[sb.cuda_stream])[0]
    torch.cuda.synchronize()
    for k, (u, v) in enumerate(zip(ra, solo_a)):
        _same(u, v, f"group: A on stream A, output {k}")
    for k, (u, v) in enumerate(zip(rb, solo_b)):
        _same(u, v, f"group: B on stream B, output {k}")


# ------------------------------------------------------------------------------------------ 3. Gram calls are ordered across streams
@pytest.mark.parametrize("b_on", ["device", "host"])
@pytest.mark.parametrize("name", ["c6_fused_folded", "c6_friction_every_joint", "k9_general_pipeline"])
def test_gram_calls_are_ordered_across_streams(name, b_on, torch, gate):
    d, ch, comps, _, _, _, _ = _gram_case(name)
    n_in = d.n_inputs
    hA, A = _uniform(torch, n_in, 100_003, 41)
    hB, B = _uniform(torch, n_in, 30_011, 42)
    torch.cuda.synchronize()
    # solo runs first: they also build the run-time specialised kernel and size the workspace, so nothing below blocks the host
    solo_a = [_np(v) for v in _dev_gram(ch, comps, A, None)]
    solo_b = [_np(v) for v in _dev_gram(ch, comps, B, None)] if b_on == "device" else [v.copy() for v in ch.regressorGram(*hB)]
    torch.cuda.synchronize()
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    t0, gated, b_done = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    with torch.cuda.stream(sa):
        t0.record()
        gate(0.4)
        gated.record()
        ra = _dev_gram(ch, comps, A, None)
    if b_on == "device":
        with torch.cuda.stream(sb):
            rb = _dev_gram(ch, comps, B, None)
            b_done.record()
        time.sleep(0.1)
        if not gated.query():  # the enqueue returned while the gate still runs (an enqueue may wait for the stream, e.g. a pageable copy)
            assert not b_done.query(), f"{name}: the Gram call on stream B finished while the call before it on stream A waits behind the gate"
        torch.cuda.synchronize()
        ms_gate, ms_b = t0.elapsed_time(gated), t0.elapsed_time(b_done)
        assert ms_b >= ms_gate, f"{name}: the Gram call on stream B finished {ms_b:.1f} ms after the gate started, before its end ({ms_gate:.1f} ms)"
    else:
        rb = ch.regressorGram(*hB)
        assert gated.query(), f"{name}: the host Gram entry returned while a device Gram call of the handle was still queued"
    torch.cuda.synchronize()
    for k, (u, v) in enumerate(zip(ra, solo_a)):
        _same(u, v, f"{name}: gated A, output {k}")
    for k, (u, v) in enumerate(zip(rb, solo_b)):
        _same(u, v, f"{name}: B ({b_on}), output {k}")


# ------------------------------------------------------------------------------------------ 4. a model change waits for work in flight
def test_input_selection_waits_for_queued_calls(torch, gate):
    """n_inputs stays the same (the inputs are reversed), so that every read stays in bounds whatever the order of events"""
    from rosdyn_b200.chain import Chain
    d6, d64 = fixtures.by_name("c6"), desc("unf64_rev")
    ch6, ch64 = Chain(d6), Chain(d64)
    r6, r64 = ch6.getActiveJointsName()[::-1], ch64.getActiveJointsName()[::-1]
    new6, new64 = copy.deepcopy(d6), copy.deepcopy(d64)
    new6.set_input_joints(r6)
    new64.set_input_joints(r64)
    ch6n, ch64n = Chain(new6), Chain(new64)
    _, x6 = _uniform(torch, 6, 20011, 51)
    _, x64 = _uniform(torch, d64.n_inputs, 2003, 52)
    goal = torch.tensor(np.random.RandomState(53).uniform(-1, 1, (6, 4099)), device="cuda")
    target = ch6.kinematics(goal, want=("T_tool",))["T_tool"].clone()
    seed = goal + torch.tensor(np.random.RandomState(54).uniform(-0.3, 0.3, (6, 4099)), device="cuda")
    lim = np.full(6, 2.5)

    def calls(c6, c64):
        return {"ik": c6.computeLocalIk(target, seed, -lim, lim, toll=1e-9, max_iter=30),
                "kinematics64": tuple(c64.kinematics(x64[0], x64[1], want=("T_tool", "jacobian", "twist")).values()),
                "torque64": (c64.getJointTorque(*x64),),
                "gram_folded": c6.regressorGram(*x6)}
    torch.cuda.synchronize()
    old = {k: [_np(v) for v in r] for k, r in calls(ch6, ch64).items()}
    new = {k: [_np(v) for v in r] for k, r in calls(ch6n, ch64n).items()}
    for k in old:
        assert any(not np.array_equal(u, v) for u, v in zip(old[k], new[k])), f"{k}: the reversed input order must change the result"
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        gate(0.4)
        gated = calls(ch6, ch64)
    assert ch6.setInputJointsName(r6) and ch64.setInputJointsName(r64)
    with torch.cuda.stream(sb):
        after = calls(ch6, ch64)
    torch.cuda.synchronize()
    for k in old:
        for j, (u, v) in enumerate(zip(gated[k], old[k])):
            _same(u, v, f"{k} queued before the input change, output {j}")
        for j, (u, v) in enumerate(zip(after[k], new[k])):
            _same(u, v, f"{k} issued after the input change, output {j}")


# -------------------------------------------------------------------------------------- 5. const entries run concurrently on one handle
def test_const_entries_run_concurrently_on_one_handle(torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name("c6")
    ch = Chain(d)
    x = _big(6, 1_000_003, 0x5EED0000 + 61)

    def kin():
        return tuple(ch.kinematics(*x[:3], want=KIN).values())

    def reg():
        return ch.getRegressor(*x[:3], with_torque=True)

    def fd():
        return ch.getJointAcceleration(x[0], x[1], x[3], with_info=True)
    torch.cuda.synchronize()
    solo = [[_np(v) for v in f()] for f in (kin, reg, fd)]
    streams = [torch.cuda.Stream() for _ in range(3)]
    res = []
    for s, f in zip(streams, (kin, reg, fd)):
        with torch.cuda.stream(s):
            res.append(f())
    torch.cuda.synchronize()
    for name, r, ref in zip(("kinematics", "regressor", "forward dynamics"), res, solo):
        for k, (u, v) in enumerate(zip(r, ref)):
            _same(u, v, f"{name} on its own stream, output {k}")
