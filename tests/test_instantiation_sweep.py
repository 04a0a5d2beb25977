"""Every compiled instantiation of the hot-path kernels against the CPU oracle.

Each kernel template is instantiated per chain size (and per output mask, per all-revolute variant, per component width), and every
instantiation is separate SASS with its own register allocation, tile mapping and loop bounds.  The chain family below is built so that
every dispatch key of the launchers is reached:

* kinematics walker ``kin_kernel<NJ, MASK, NP>``: NJ = 1..8 (fixed joints included) x no-prismatic or not x the 7 compiled output masks,
  and the generic kernel above 8;
* regressor walker ``dyn_kernel<NJ, REGRESSOR, false, REC>`` on the unfolded chain, SoA and Eigen-record layouts;
* torque / inertia / forward-dynamics walkers on the folded chain, K = 1..8 moving inputs x all-revolute or not, generic above 8;
* wrench / link Jacobian (``aux_kernel``), fast and generic;
* fused Gram ``gram_fused_kernel<K, .., REV, 0>``, K = 1..7, run-time specialised (NVRTC) and precompiled twins;
* extended Gram ``gram_fused_kernel<K, .., REV, XC>``, K = 1..7, XC = 2, 4, 8 component columns on the widest joint;
* the general Gram pipeline (gram.cu): K >= 8, no moving joint, and the component sets the one-pass kernel refuses.

The CPU test recomputes each case's dispatch key from its descriptor with the launchers' rules and fails when the family stops covering
one of them.  Tolerance: the project contract maxabs(x - ref) <= 1e-10 max(maxabs(ref), 1), applied per output plane (per link, per joint
row, per Jacobian column), and for the normal equations per entry against its Cauchy-Schwarz scale sqrt(G_ii G_jj)."""
import math

import numpy as np
import pytest

from conftest import RTOL
from rosdyn_b200 import fixtures
from rosdyn_b200.descriptor import FIXED, PRISMATIC, REVOLUTE

KIN = ("T_tool", "T_links", "jacobian", "twist", "dtwist", "dtwist_lin", "dtwist_nonlin", "ddtwist", "ddtwist_lin", "ddtwist_nonlin",
       "torque")
BIT = {k: 1 << i for i, k in enumerate(KIN)}  # rdb_kinematics_out field -> K_* bit (chain_dev.h)
K_ALL = (1 << len(KIN)) - 1


def _mask(*fields):
    m = 0
    for f in fields:
        m |= BIT[f]
    return m


# the compiled output combinations of launch_kin (kernels.cu), in the order it tries them
KM_POSE = _mask("T_tool", "T_links")
KM_POSE_JAC = KM_POSE | BIT["jacobian"]
KM_VEL = KM_POSE_JAC | BIT["twist"]
KM_CFG2 = _mask("T_tool", "jacobian", "twist", "dtwist", "torque")
KM_JERK = _mask("twist", "dtwist", "ddtwist")
KM_ACC = KM_VEL | _mask("dtwist", "dtwist_lin", "dtwist_nonlin")
MASKS = {"pose": KM_POSE, "pose_jac": KM_POSE_JAC, "vel": KM_VEL, "cfg2": KM_CFG2, "jerk": KM_JERK, "acc": KM_ACC, "all": K_ALL}


def launched_mask(want):
    """The mask launch_kin compiles for a request: the first compiled combination that covers it."""
    m = _mask(*want)
    for name in ("pose", "pose_jac", "vel", "cfg2", "jerk", "acc"):
        if m & ~MASKS[name] == 0:
            return name
    return "all"


# every compiled mask requested exactly, and odd subsets that launch_kin rounds up to one of them
KIN_WANTS = [tuple(k for k in KIN if MASKS[m] & BIT[k]) for m in MASKS] + [("dtwist_lin",), ("torque", "T_links"), ("twist",),
                                                                            ("ddtwist_lin", "jacobian")]


# ---------------------------------------------------------------------------------------------------------------------------- chains
def _chain(seed, types, axis_z=False):
    """fixtures.random_chain (oblique axes, random frames, full inertias) with the joint types set explicitly; axis_z: every revolute
    joint turns about +z of its own frame, so that nothing is rotated when the chain is folded."""
    d = fixtures.random_chain(seed, len(types), p_prismatic=0.0, p_fixed=0.0)
    for j, t in zip(d.joints, types):
        j.type = t
        if axis_z and t == REVOLUTE:
            j.axis = (0.0, 0.0, 1.0)
    d.set_default_inputs()
    return d


def unfolded(nj, variant):
    """nj chain joints; from 3 on one interior fixed joint; "pri": the last joint prismatic."""
    types = [REVOLUTE] * nj
    if nj >= 3:
        types[nj // 2] = FIXED
    if variant == "pri":
        types[-1] = PRISMATIC
    d = _chain(7000 + 3 * nj + (variant == "pri"), types)
    d.name = f"unf{nj}_{variant}"
    return d


def folded(k, kind, shape):
    """k moving input joints.  shape "tool": a leading fixed joint and a massive fixed tool (the fold is not the identity); "plain": no
    fixed joint and every revolute axis on +z (nothing to fold).  kind "mix": the middle moving joint prismatic."""
    moving = [REVOLUTE] * k
    if kind == "mix":
        moving[k // 2] = PRISMATIC
    if shape == "tool":
        d = _chain(8000 + 5 * k + (kind == "mix"), [FIXED] + moving + [FIXED])
    else:
        d = _chain(8500 + 5 * k + (kind == "mix"), moving, axis_z=True)
    d.name = f"fold{k}_{kind}_{shape}"
    return d


def reversed_inputs():
    """3 moving revolute joints fed by the inputs in reverse order"""
    d = folded(3, "rev", "tool")
    d.set_input_joints([j.name for j in d.joints if j.type != FIXED][::-1])
    d.name = "k3_rev_reversed"
    return d


def unlisted_input():
    """7 moving joints (the 4th prismatic), the 2nd of them not an input: it stays at q = 0 and folds away (K = 6)"""
    d = folded(7, "mix", "tool")
    names = [j.name for j in d.joints if j.type != FIXED]
    d.set_input_joints(names[:1] + names[2:])
    d.name = "k6_mix_unlisted"
    return d


def axis_aligned():
    """2 revolute joints with coordinate axes, signed-permutation joint frames, axis-aligned offsets and inertias: the folded constants are
    exact zeros and ones, which the run-time specialised generator drops"""
    from rosdyn_b200.descriptor import ChainDesc, JointDesc, LinkDesc
    J = [JointDesc("a0", REVOLUTE, (0.0, 0.0, 0.25), (0, 0, 1, 0, 1, 0, -1, 0, 0), (0.0, 1.0, 0.0)),
         JointDesc("a1", REVOLUTE, (0.0, 0.3, 0.0), (1, 0, 0, 0, 0, -1, 0, 1, 0), (-1.0, 0.0, 0.0))]
    L = [LinkDesc("base", 1.0), LinkDesc("l1", 3.0, (0.0, 0.0, 0.1), inertia=(0.03, 0.0, 0.0, 0.02, 0.0, 0.01)),
         LinkDesc("l2", 1.5, (0.1, 0.0, 0.0), inertia=(0.01, 0.0, 0.0, 0.02, 0.0, 0.025))]
    return ChainDesc(J, L, fixtures.GRAVITY, name="k2_rev_axis_aligned")


def unfed_input(k, kind):
    """folded(k, kind, "tool") with one more input that no chain joint feeds (a name not in the chain): inputs_cover_all is false"""
    d = folded(k, kind, "tool")
    d.set_input_joints([j.name for j in d.joints if j.type != FIXED] + ["no_such_joint"])
    d.name = f"k{k}_{kind}_unfed_input"
    return d


def no_moving_joint():
    """one input, fed by no chain joint: K = 0"""
    d = folded(2, "rev", "tool")
    d.set_input_joints(["no_such_joint"])
    d.name = "k0_no_moving_joint"
    return d


CASES = {}
for _nj in list(range(1, 10)) + [64]:
    for _v in ("rev", "pri"):
        CASES[f"unf{_nj}_{_v}"] = (lambda nj=_nj, v=_v: unfolded(nj, v))
for _k in range(1, 10):
    for _kind in ("rev", "mix"):
        for _shape in ("tool", "plain"):
            CASES[f"fold{_k}_{_kind}_{_shape}"] = (lambda k=_k, kind=_kind, shape=_shape: folded(k, kind, shape))
for _kind in ("rev", "mix"):
    CASES[f"fold64_{_kind}_plain"] = (lambda kind=_kind: folded(64, kind, "plain"))
CASES["k3_rev_reversed"] = reversed_inputs
CASES["k6_mix_unlisted"] = unlisted_input
CASES["k2_rev_axis_aligned"] = axis_aligned
CASES["k3_rev_unfed_input"] = lambda: unfed_input(3, "rev")
CASES["k9_rev_unfed_input"] = lambda: unfed_input(9, "rev")
CASES["k0_no_moving_joint"] = no_moving_joint

UNFOLDED = [f"unf{nj}_{v}" for nj in list(range(1, 10)) + [64] for v in ("rev", "pri")]
UNFOLDED_SMALL = [c for c in UNFOLDED if not c.startswith("unf64")]
EXTRA = ["k3_rev_reversed", "k6_mix_unlisted", "k2_rev_axis_aligned", "k3_rev_unfed_input"]
FOLDED = [f"fold{k}_{kind}_{s}" for k in range(1, 10) for kind in ("rev", "mix") for s in ("tool", "plain")] + \
         ["fold64_rev_plain", "fold64_mix_plain"] + EXTRA
GRAM_FUSED = [c for c in FOLDED if c.startswith("fold") and int(c[4:c.index("_")]) <= 7] + EXTRA
# extended model: (case, widest component set on one joint); XC 2 and 4 at every K on the generic generator, at K = 1, 2 on the REV one
EXT_RUNS = [(f"fold{k}_mix_tool", xc) for k in range(1, 8) for xc in (2, 4, 8)] + \
           [(f"fold{k}_rev_tool", 8) for k in range(1, 8)] + [(f"fold{k}_rev_tool", xc) for k in (1, 2) for xc in (2, 4)] + \
           [("k3_rev_unfed_input", 8)]
# general pipeline: (case, component set); None = rigid-body normal equations
GENERAL_RUNS = [(f"fold{k}_{kind}_{s}", None) for k in (8, 9) for kind in ("rev", "mix") for s in ("tool", "plain")] + \
               [("k9_rev_unfed_input", None), ("k0_no_moving_joint", None), ("unf64_rev", None),
                ("fold3_mix_tool", "nine_columns"), ("k3_rev_unfed_input", "unfed"), ("fold9_mix_tool", 8)]


def desc(name):
    return CASES[name]()


# ------------------------------------------------------------------------------------------------------------- dispatch keys (host)
def fold_k(d):
    """moving joints of the folded chain: chain joints fed by an input (fold.cpp counts every joint with an input index)"""
    return sum(1 for j in d.joints if j.input_index >= 0)


def fold_rev(d):
    return all(j.type == REVOLUTE for j in d.joints if j.input_index >= 0)


def kin_key(d, want):
    """launch_kin_mask: NJ of the unfolded chain (generic above 8), no prismatic joint anywhere in it, the mask picked for the request"""
    nj = d.n_joints
    return (nj if nj <= 8 else "generic", all(j.type != PRISMATIC for j in d.joints), launched_mask(want))


def walker_key(d):
    """launch_dyn_mode for torque / inertia / FD: the folded chain's K (generic above 8), all-revolute specialisation"""
    k = fold_k(d)
    return (k if 1 <= k <= 8 else "generic", fold_rev(d))


def components(d, spec):
    """component list [(type, input index, min_velocity, max_velocity)] of a named set.  int spec: widest joint carries `spec` columns
    (8 = friction2 + friction2 + friction1, 4 = friction1 + spring, 2 = spring), the last moving input a friction1 (2 columns);
    "nine_columns": 3 x friction2 on one joint; "unfed": a friction1 on the input no chain joint feeds."""
    ins = sorted(j.input_index for j in d.joints if j.input_index >= 0)
    lo, hi = 0.05, 0.7
    if spec == "nine_columns":
        return [(2, ins[0], lo, hi)] * 3
    if spec == "unfed":
        fed = set(ins)
        free = [i for i in range(d.n_inputs) if i not in fed]
        return [(1, ins[0], lo, hi), (1, free[0], lo, hi)]
    wide = {8: [(2, ins[0], lo, hi), (2, ins[0], 0.1, 0.9), (1, ins[0], lo, hi)], 4: [(1, ins[0], lo, hi), (3, ins[0], 0.0, 0.0)],
            2: [(3, ins[0], 0.0, 0.0)]}[spec]
    return wide + ([(1, ins[-1], 0.02, 0.5)] if len(ins) > 1 else [])


def ext_xc(d, comps):
    """launch_gram_fused_ext: XC from the widest joint's component columns, or None when the one-pass kernel refuses the set"""
    k = fold_k(d)
    fed = {j.input_index for j in d.joints if j.input_index >= 0}
    cols = {}
    for t, i, _, _ in comps:
        if i not in fed:
            return None
        cols[i] = cols.get(i, 0) + (3 if t == 2 else 2)
    w = max(cols.values())
    if not 1 <= k <= 7 or w > 8:
        return None
    return 2 if w <= 2 else (4 if w <= 4 else 8)


def gram_path(d, comps=None):
    """launch_gram: "fused" or the reason the general pipeline runs"""
    k = fold_k(d)
    if k > 7:
        return "more than 7 moving joints"
    if k < 1:
        return "no moving joint"
    if comps and ext_xc(d, comps) is None:
        return "refused component set"
    return "fused"


def test_family_covers_every_instantiation():
    """The dispatch keys the sweep reaches, recomputed from the descriptors with the launchers' rules: trimming a case fails here."""
    kin = {kin_key(desc(c), w) for c in UNFOLDED for w in KIN_WANTS}
    need = {(nj, np_, m) for nj in range(1, 9) for np_ in (True, False) for m in MASKS}
    assert need <= kin, sorted(need - kin, key=str)
    assert {("generic", True), ("generic", False)} <= {k[:2] for k in kin}
    rec = {desc(c).n_joints for c in UNFOLDED_SMALL}
    assert set(range(1, 9)) <= rec and max(rec) > 8  # regressor: REC instantiations and the generic kernel
    walk = {walker_key(desc(c)) for c in FOLDED}
    need = {(k, r) for k in range(1, 9) for r in (True, False)}
    assert need <= walk, sorted(need - walk, key=str)
    assert {("generic", True), ("generic", False)} <= walk
    fused = {(fold_k(desc(c)), fold_rev(desc(c))) for c in GRAM_FUSED}
    assert all(gram_path(desc(c)) == "fused" for c in GRAM_FUSED)
    need = {(k, r) for k in range(1, 8) for r in (True, False)}
    assert need <= fused, sorted(need - fused)
    ext = set()
    for c, xc in EXT_RUNS:
        d = desc(c)
        got = ext_xc(d, components(d, xc))
        assert got == xc, (c, xc, got)
        ext.add((fold_k(d), fold_rev(d), got))
    assert {(k, x) for k in range(1, 8) for x in (2, 4, 8)} <= {(k, x) for k, _, x in ext}
    assert {(k, r, 8) for k in range(1, 8) for r in (True, False)} <= ext
    general = {}
    for c, spec in GENERAL_RUNS:
        d = desc(c)
        why = gram_path(d, None if spec is None else components(d, spec))
        assert why != "fused", c
        general.setdefault(why, set()).add(fold_k(d))
    assert {8, 9} <= general["more than 7 moving joints"] and max(general["more than 7 moving joints"]) >= 60
    assert general["no moving joint"] == {0}
    refused = {spec for c, spec in GENERAL_RUNS if spec in ("nine_columns", "unfed")}
    assert refused == {"nine_columns", "unfed"} and "refused component set" in general
    # the fold is exercised both ways, with a massive rigid tool and with nothing to fold
    assert any(desc(c).joints[-1].type == FIXED and desc(c).links[-1].mass > 0 for c in GRAM_FUSED)
    assert any(all(j.type != FIXED for j in desc(c).joints) for c in GRAM_FUSED)


def test_case_names_state_their_shape():
    for c in UNFOLDED:
        d = desc(c)
        assert d.name == c and d.n_joints == int(c[3:c.index("_")])
        assert (c.endswith("_pri")) == any(j.type == PRISMATIC for j in d.joints)
    for c in FOLDED:
        d = desc(c)
        assert d.name == c
        if c.startswith("fold"):
            assert fold_k(d) == int(c[4:c.index("_")]) and fold_rev(d) == ("_rev_" in c)
        else:
            assert fold_k(d) == int(c[1]) and fold_rev(d) == ("_rev_" in c)


# ------------------------------------------------------------------------------------------------------- oracle self-checks (host)
def _inputs(n_in, n, seed):
    rng = np.random.RandomState(seed)
    return rng.uniform(-np.pi, np.pi, (n_in, n)), rng.uniform(-2, 2, (n_in, n)), rng.uniform(-5, 5, (n_in, n))


@pytest.mark.parametrize("name", ["unf1_pri", "unf2_rev", "unf9_pri", "unf64_rev", "fold1_mix_tool", "fold64_mix_plain", "k6_mix_unlisted",
                                  "k3_rev_reversed", "k2_rev_axis_aligned", "k3_rev_unfed_input", "k0_no_moving_joint"])
def test_oracle_is_consistent_on_the_family(name):
    """The references the GPU tests use agree with each other on these shapes: Phi pi_nom == tau, M ddq + h == tau, the long-double
    normal equations == the numpy contraction of the regressor, and the forward-dynamics composition solves tau back to ddq."""
    from oracle.oracle import OracleChain
    from test_forward_dynamics import oracle_fd
    d = desc(name)
    oc = OracleChain(d)
    n_in, P = d.n_inputs, 10 * d.n_joints
    n = 40
    q, dq, ddq = _inputs(n_in, n, 3)
    phi, tau = oc.regressor_torque(q, dq, ddq)
    Phi = phi.reshape(P, n_in, n)
    pi = oc.nominal_parameters()
    tscale = max(np.max(np.abs(tau)), 1.0)
    assert np.max(np.abs(np.einsum("cri,c->ri", Phi, pi) - tau)) <= 1e-10 * tscale
    _, h = oc.regressor_torque(q, dq, np.zeros_like(ddq))
    M = oc.inertia(q).reshape(n_in, n_in, n)  # plane col * n_in + row
    assert np.max(np.abs(np.einsum("cri,ci->ri", M, ddq) + h - tau)) <= 1e-10 * tscale
    Gr, br, ttr = oc.gram(q, dq, ddq)
    X = Phi.reshape(P, -1)
    gs = max(np.max(np.abs(Gr)), 1e-300)
    assert np.max(np.abs(X @ X.T - Gr)) <= 1e-12 * gs and abs(np.sum(tau * tau) - ttr) <= 1e-12 * max(ttr, 1.0)
    fed = [j.input_index for j in d.joints if j.input_index >= 0]
    if fed:
        acc = oracle_fd(d, q, dq, tau)
        assert np.max(np.abs(acc[fed] - ddq[fed])) <= 1e-7 * np.max(np.abs(ddq)), "M(q) too ill-conditioned for an FD comparison"


# ----------------------------------------------------------------------------------------------------------------- GPU helpers
def _np(t):
    return t.detach().cpu().numpy()


def assert_planes(x, ref, rows, what, rtol=RTOL):
    """x, ref: [planes * rows, N] (or [planes * rows]); every plane of `rows` rows within rtol * max(maxabs(ref plane), 1)"""
    x, ref = np.asarray(x, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    assert x.shape == ref.shape, (what, x.shape, ref.shape)
    if x.size == 0:
        return
    npl = ref.shape[0] // rows
    e = np.abs(x - ref).reshape(npl, -1).max(axis=1)
    s = np.maximum(np.abs(ref).reshape(npl, -1).max(axis=1), 1.0)
    bad = np.nonzero(~(e <= rtol * s))[0]
    assert bad.size == 0, f"{what}: {bad.size} of {npl} planes ({rows} rows each) off, worst plane {bad[np.argmax((e / s)[bad])]}: " \
                          f"rel err {np.max((e / s)[bad]):.3e} > {rtol:.0e}"


def assert_gram(G, b, tt, Gr, br, ttr, what, rtol=1e-10):
    """Normal equations against a reference: every entry within rtol of its Cauchy-Schwarz scale sqrt(Gr_ii Gr_jj), b_i within rtol of
    sqrt(Gr_ii tau^T tau), tau^T tau within rtol, G symmetric bit for bit, and the project contract on the whole matrix.

    The scales have a floor for the columns that are zero in exact arithmetic (the first moving link's inertia products, m c_z and m; the
    kernels keep them exactly zero, the reference leaves rounding residue there).  A residue of c ulps of the largest entry of each
    regressor row gives |Gr_ij| <= c eps sqrt(tr(Gr) Gr_jj) and |br_i| <= c eps sqrt(tr(Gr) tau^T tau) (Cauchy-Schwarz over the rows), which
    does not average out at n = 1.  The floors are 1e-4 sqrt(tr(Gr) max(Gr_ii, Gr_jj)) and 1e-4 sqrt(tr(Gr) tau^T tau), i.e. residues up to
    c = 45 pass; they exceed sqrt(Gr_ii Gr_jj) only where Gr_ii < 1e-8 tr(Gr), so every column with weight keeps the full check."""
    G, b, Gr, br = (np.asarray(x, dtype=np.float64) for x in (G, b, Gr, br))
    tt, ttr = float(np.asarray(tt).reshape(-1)[0]), float(ttr)
    assert np.isfinite(G).all() and np.isfinite(b).all() and math.isfinite(tt), what
    assert np.array_equal(G, G.T), f"{what}: gram not symmetric"
    dg = np.clip(np.diag(Gr), 0.0, None)
    tr = dg.sum()
    sc = np.maximum(np.sqrt(np.outer(dg, dg)), 1e-4 * np.sqrt(tr * np.maximum.outer(dg, dg)))
    e = np.abs(G - Gr)
    bad = np.argwhere(~(e <= rtol * sc))
    assert bad.size == 0, f"{what}: {len(bad)} gram entries off their Cauchy-Schwarz scale, e.g. {tuple(bad[0])}: " \
                          f"{G[tuple(bad[0])]!r} vs {Gr[tuple(bad[0])]!r}"
    assert np.max(e, initial=0.0) <= rtol * max(np.max(np.abs(Gr), initial=0.0), 1.0), what
    sb = np.maximum(np.sqrt(dg * ttr), 1e-4 * math.sqrt(tr * ttr))
    bad = np.nonzero(~(np.abs(b - br) <= rtol * sb))[0]
    assert bad.size == 0, f"{what}: rhs entries {bad[:8]} off: {b[bad[0]]!r} vs {br[bad[0]]!r}"
    assert abs(tt - ttr) <= rtol * ttr, f"{what}: tau_sq {tt!r} vs {ttr!r}"


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _dev(torch, *xs):
    return [torch.tensor(np.ascontiguousarray(x), device="cuda") for x in xs]


def _gpu_inputs(torch, n_in, n, seed):
    h = _inputs(n_in, n, seed)
    return h, _dev(torch, *h)


# ------------------------------------------------------------------------------------------------------------------ kinematics
@pytest.mark.gpu
@pytest.mark.parametrize("name", UNFOLDED)
def test_kinematics_every_mask(name, torch):
    """Each compiled mask, and odd subsets launch_kin rounds up, against the oracle per plane, and bit for bit against the K_ALL call."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    from test_round2_gpu import _planted_inputs
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in, nL = d.n_inputs, d.n_joints + 1
    rows = {"T_tool": 12, "T_links": 12, "jacobian": 6, "torque": 1}
    big = 4099 if d.n_joints <= 9 else 515
    hq = _planted_inputs(n_in, big, 0x5EED0000 + d.n_joints)
    for sl in (slice(0, big), slice(9, 10)):  # every planted edge sample in a ragged batch, and n = 1
        h = [np.ascontiguousarray(x[:, sl]) for x in hq]
        x = _dev(torch, *h)
        ref = oc.kinematics(*h, nthreads=0)
        full = {k: _np(v) for k, v in ch.kinematics(*x, want=KIN).items()}
        n = h[0].shape[1]
        for k in KIN:
            assert_planes(full[k], ref[k], rows.get(k, 6), f"{name} n={n} K_ALL:{k}")
        for want in KIN_WANTS:
            out = ch.kinematics(*x, want=want)
            assert set(out) == set(want)
            for k, v in out.items():
                v = _np(v)
                assert_planes(v, ref[k], rows.get(k, 6), f"{name} n={n} {launched_mask(want)}{want}:{k}")
                assert np.array_equal(v, full[k]), f"{name} n={n}: {k} of mask {launched_mask(want)} differs from K_ALL by " \
                                                   f"{np.max(np.abs(v - full[k])):.3e}"
    assert nL == len(ch.getLinksName())


# ------------------------------------------------------------------------------------------------------------------- regressor
@pytest.mark.gpu
@pytest.mark.parametrize("name", UNFOLDED_SMALL)
def test_regressor_soa_and_records(name, torch):
    """SoA regressor against the oracle per (joint row, link block), exact structural zeros; the Eigen-record layout (REC instantiation)
    bit for bit against SoA."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in, P = d.n_inputs, 10 * d.n_joints
    for n in (4099, 1):
        h, x = _gpu_inputs(torch, n_in, n, 40 + n)
        rphi, rtau = oc.regressor_torque(*h, nthreads=0)
        phi, tau = ch.getRegressor(*x, with_torque=True)
        planes = _np(phi.transpose(0, 1).reshape(P * n_in, n))
        # plane index c * n_in + r: group by (link block, joint row)
        blk = planes.reshape(d.n_joints, 10, n_in, n).transpose(0, 2, 1, 3).reshape(-1, n)
        rblk = rphi.reshape(d.n_joints, 10, n_in, n).transpose(0, 2, 1, 3).reshape(-1, n)
        assert_planes(blk, rblk, 10, f"{name} n={n}: regressor")
        assert_planes(_np(tau), rtau, 1, f"{name} n={n}: torque of the regressor pass")
        Phi = planes.reshape(P, n_in, n)
        for j, jd in enumerate(d.joints):
            if jd.input_index >= 0:
                assert np.all(Phi[:10 * j, jd.input_index, :] == 0.0), f"{name}: structural zeros of joint {j} must be exact"
        rec = ch.dynamics(*x, want=("regressor", "torque"), layout="eigen")
        assert torch.equal(rec["regressor"].permute(1, 2, 0), phi), f"{name} n={n}: record layout != SoA"
        assert torch.equal(rec["torque"].transpose(0, 1), tau), f"{name} n={n}: record torque != SoA"


# ---------------------------------------------------------------------------------------------------- torque, inertia, FD
@pytest.mark.gpu
@pytest.mark.parametrize("name", FOLDED)
def test_torque_inertia_forward_dynamics(name, torch):
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    from test_forward_dynamics import oracle_fd
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in = d.n_inputs
    n = 3001 if d.n_joints <= 11 else 257
    h, x = _gpu_inputs(torch, n_in, n, 60)
    _, rtau = oc.regressor_torque(*h, nthreads=0)
    tau = ch.getJointTorque(*x)
    assert_planes(_np(tau), rtau, 1, f"{name}: torque")
    M = _np(ch.getJointInertia(x[0]).transpose(0, 1).reshape(n_in * n_in, n))
    assert_planes(M, oc.inertia(h[0], nthreads=0), n_in, f"{name}: inertia (per column)")
    rng = np.random.RandomState(61)
    tau_a = rng.uniform(-20, 20, (n_in, n))
    ddq, info = ch.getJointAcceleration(x[0], x[1], _dev(torch, tau_a)[0], with_info=True)
    assert int(info.abs().sum()) == 0, f"{name}: info != 0"
    # ddq = M^-1 (tau - h): a backward-stable solve leaves about cond(M) eps relative.  M of the 64-joint chains reaches cond 7.6e5 on these
    # samples (the oracle's own round trip is off by 4e-11 there), so they get 1e-9; every other case has cond <= 1.4e4 and keeps RTOL
    tol = RTOL if fold_k(d) <= 9 else 1e-9
    assert_planes(_np(ddq), oracle_fd(d, h[0], h[1], tau_a), 1, f"{name}: forward dynamics", tol)
    back = _np(ch.getJointAcceleration(x[0], x[1], tau))
    fed = [j.input_index for j in d.joints if j.input_index >= 0]
    assert_planes(back[fed], h[2][fed], 1, f"{name}: forward dynamics of the device torque", tol)


# ---------------------------------------------------------------------------------------------------- wrench, link Jacobian
@pytest.mark.gpu
@pytest.mark.parametrize("name", UNFOLDED_SMALL)
def test_wrench_and_link_jacobian(name, torch):
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in, nL = d.n_inputs, d.n_joints + 1
    n = 2049
    h, x = _gpu_inputs(torch, n_in, n, 80)
    ext = np.random.RandomState(81).normal(size=(6 * nL, n)) * 10.0
    tau_ref, w_ref = oc.wrench(*h, ext)
    w, tau = ch.getWrench(*x, _dev(torch, ext)[0].reshape(nL, 6, n), with_torque=True)
    assert_planes(_np(tau), tau_ref, 1, f"{name}: torque with external wrenches")
    assert_planes(_np(w.reshape(-1, n)), w_ref, 6, f"{name}: wrenches (per link)")
    names = ch.getLinksName()
    for link in sorted({0, 1, nL - 1}):
        J = _np(ch.getJacobianLink(x[0], names[link]).transpose(0, 1).reshape(6 * n_in, n))
        assert_planes(J, oc.jacobian_link(h[0], link), 6, f"{name}: jacobian of link {link} (per column)")


# ------------------------------------------------------------------------------------------------------------------ fused Gram
def _both(ch, fn, monkeypatch):
    from test_gram_specialised import _both as both
    return both(ch, fn, monkeypatch)


def _oracle_gram(oc, h, tau=None):
    from test_round2_gpu import _oracle_gram_parallel
    if h[0].shape[1] < 4096:
        return oc.gram(*h, tau)
    return _oracle_gram_parallel(oc, *h, tau=tau)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GRAM_FUSED)
def test_fused_gram(name, torch, monkeypatch):
    """Every CTA takes several 32-sample groups and ends ragged (20 011 samples on 148 SMs), plus n = 1 and 31; computed and measured
    torques; accumulation adds exactly; REV chains: the NVRTC and the precompiled kernel bit for bit."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    rev = fold_rev(d)
    n_in = d.n_inputs
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    big = 4 * 32 * sm + 32 * 8 + 11
    for n in (big, 1, 31):
        h, x = _gpu_inputs(torch, n_in, n, 100 + n)
        tm = np.random.RandomState(n).uniform(-50, 50, (n_in, n))
        for t_h in (None, tm):
            t_d = None if t_h is None else _dev(torch, t_h)[0]
            what = f"{name} n={n} tau={'measured' if t_h is not None else 'computed'}"
            if rev:
                a, b, ia, ib = _both(ch, lambda: ch.regressorGram(*x, tau_meas=t_d), monkeypatch)
                assert ia[0] == 1 and ib[0] == 0, (ia, ib)
                for u, v, k in zip(a, b, ("gram", "rhs", "tau_sq")):
                    assert np.array_equal(u, v), f"{what}: {k} of the NVRTC and precompiled kernels differ by {np.max(np.abs(u - v)):.3e}"
                G, bb, tt = a
            else:
                G, bb, tt = (_np(v) for v in ch.regressorGram(*x, tau_meas=t_d))
                assert ch.gramKernelInfo()[0] == 0
            assert_gram(G, bb, tt, *_oracle_gram(oc, h, t_h), what)
            if n == big:  # accumulate: adds the second call's result onto the first exactly
                out = tuple(torch.tensor(v, device="cuda") for v in (G, bb, tt))
                ch.regressorGram(*x, tau_meas=t_d, out=out)
                for o, v, k in zip(out, (G, bb, tt), ("gram", "rhs", "tau_sq")):
                    assert np.array_equal(_np(o), v + v), f"{what}: accumulated {k}"


# --------------------------------------------------------------------------------------------------------------- extended Gram
def _ext_reference(d, oc, h, comps, tau=None):
    from oracle import oracle
    n_in, P = d.n_inputs, 10 * d.n_joints
    n = h[0].shape[1]
    phi, rtau = oc.regressor_torque(*h, nthreads=0)
    X = phi.reshape(P, n_in, n)
    if comps:
        pc = sum(3 if t == 2 else 2 for t, _, _, _ in comps)
        X = np.concatenate([X, oracle.components_regressor(comps, n_in, h[0], h[1]).reshape(pc, n_in, n)])
    t = rtau if tau is None else tau
    X2 = X.reshape(X.shape[0], -1)
    return X2 @ X2.T, X2 @ t.reshape(-1), float(np.sum(t * t))


def _set_components(ch, comps):
    tn = {1: "friction1", 2: "friction2", 3: "spring"}
    return ch.setComponents([{"type": tn[t], "joint": j, "min_velocity": lo, "max_velocity": hi} for t, j, lo, hi in comps])


@pytest.mark.gpu
@pytest.mark.parametrize("name,xc", EXT_RUNS)
def test_extended_gram(name, xc, torch, monkeypatch):
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    comps = components(d, xc)
    _set_components(ch, comps)
    n = 4099
    h, x = _gpu_inputs(torch, d.n_inputs, n, 200 + xc)
    h[1][:, :3] = 0.0  # omega == 0 branch of the friction columns
    x[1][:, :3] = 0.0
    if fold_rev(d):
        a, b, ia, ib = _both(ch, lambda: ch.regressorGramExt(*x), monkeypatch)
        assert ia[0] == 1 and ib[0] == 0, (ia, ib)
        for u, v in zip(a, b):
            assert np.array_equal(u, v), f"{name} XC={xc}: NVRTC and precompiled extended kernels differ by {np.max(np.abs(u - v)):.3e}"
        G, bb, tt = a
    else:
        G, bb, tt = (_np(v) for v in ch.regressorGramExt(*x))
        assert ch.gramKernelInfo()[0] == 0
    assert_gram(G, bb, tt, *_ext_reference(d, oc, h, comps), f"{name} XC={xc}")
    tm = np.random.RandomState(7).uniform(-50, 50, (d.n_inputs, n))
    G2, b2, t2 = (_np(v) for v in ch.regressorGramExt(*x, tau_meas=_dev(torch, tm)[0]))
    assert_gram(G2, b2, t2, *_ext_reference(d, oc, h, comps, tm), f"{name} XC={xc} measured torque")
    out = tuple(torch.tensor(v, device="cuda") for v in (G2, b2, t2))
    ch.regressorGramExt(*x, tau_meas=_dev(torch, tm)[0], out=out)
    for o, v, k in zip(out, (G2, b2, t2), ("gram", "rhs", "tau_sq")):
        assert np.array_equal(_np(o), v + v), f"{name} XC={xc}: accumulated {k}"


# ---------------------------------------------------------------------------------------------------------- general pipeline
def _general_chunk(d, pc=0):
    """samples per chunk of launch_gram's general pipeline (gram.cu)"""
    P, n_in = 10 * d.n_joints + pc, d.n_inputs
    return max(1024, (48 << 20) // (8 * (P * n_in + n_in))) // 128 * 128


@pytest.mark.gpu
@pytest.mark.parametrize("name,spec", GENERAL_RUNS)
def test_general_gram_pipeline(name, spec, torch):
    """Chains the fused kernels do not take: the materialised regressor and the tiled contraction, batches of 1, 127, 129 and more than
    one chunk, computed and measured torques, accumulation; gramKernelInfo() reports 2 and the cause."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc(name)
    ch, oc = Chain(d), OracleChain(d)
    n_in = d.n_inputs
    comps = None if spec is None else components(d, spec)
    pc = 0 if comps is None else _set_components(ch, comps)
    gram = ch.regressorGram if comps is None else ch.regressorGramExt
    why = {"more than 7 moving joints": "more than 7 moving joints", "no moving joint": "no moving joint",
           "refused component set": "component set"}[gram_path(d, comps)]
    big = d.n_joints > 20
    ns = (300,) if big else (1, 127, 129, _general_chunk(d, pc) + 1153)

    def ref(h, tau=None):
        if big or comps is not None:
            return _ext_reference(d, oc, h, comps or [], tau)
        return _oracle_gram(oc, h, tau)

    for n in ns:
        h, x = _gpu_inputs(torch, n_in, n, 300 + n)
        G, bb, tt = gram(*x)
        flag, reason = ch.gramKernelInfo()
        assert flag == 2 and reason.startswith("general pipeline:") and why in reason, (flag, reason)
        G, bb, tt = _np(G), _np(bb), _np(tt)
        assert_gram(G, bb, tt, *ref(h), f"{name} {spec} n={n}")
        tm = np.random.RandomState(n).uniform(-50, 50, (n_in, n))
        G2, b2, t2 = (_np(v) for v in gram(*x, tau_meas=_dev(torch, tm)[0]))
        assert_gram(G2, b2, t2, *ref(h, tm), f"{name} {spec} n={n} measured torque")
        out = tuple(torch.tensor(v, device="cuda") for v in (G, bb, tt))
        gram(*x, out=out)
        # one chunk: old + s exactly; several chunks add one after the other onto the old value
        tol = 0.0 if n <= _general_chunk(d, pc) else 1e-14
        for o, v, k in zip(out, (G, bb, tt), ("gram", "rhs", "tau_sq")):
            e = np.max(np.abs(_np(o) - 2 * v), initial=0.0)
            assert e <= tol * max(np.max(np.abs(v), initial=0.0), 1e-300), f"{name} n={n}: accumulated {k} off by {e:.3e}"


@pytest.mark.gpu
def test_kernel_info_follows_the_input_selection(torch):
    """K = 7 runs the fused kernel (1: compiled at run time); selecting the 8th moving joint too moves the chain to the general pipeline,
    and the report says so instead of keeping the fused kernel's 1."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = desc("fold8_rev_plain")
    ch = Chain(d)
    names = [j.name for j in d.joints]
    assert ch.setInputJointsName(names[:7])
    h, x = _gpu_inputs(torch, 7, 515, 400)
    ch.regressorGram(*x)
    assert ch.gramKernelInfo()[0] == 1, ch.gramKernelInfo()
    assert ch.setInputJointsName(names)
    h, x = _gpu_inputs(torch, 8, 515, 401)
    G, b, tt = ch.regressorGram(*x)
    flag, reason = ch.gramKernelInfo()
    assert flag == 2 and reason.startswith("general pipeline: more than 7 moving joints"), (flag, reason)
    assert_gram(_np(G), _np(b), _np(tt), *OracleChain(d).gram(*h), "fold8_rev_plain after the selection")
