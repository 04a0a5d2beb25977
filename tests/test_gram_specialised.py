"""Fused Gram kernels specialised at run time to the chain's constants (csrc/gram_jit.cpp): the specialised kernel must give exactly what the
precompiled kernel gives -- same operations in the same order, only the products with exact zeros dropped and those with +-1 passed through.
RDB_GRAM_JIT=0 forces the precompiled kernel on the same handle; rdb_chain_gram_kernel_info says which one ran."""
import os
import subprocess
import sys

import numpy as np
import pytest

from rosdyn_b200 import fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANDOM = {"rev_fixed_a": lambda: fixtures.random_chain(515, 7, p_prismatic=0.0, p_fixed=0.2),
          "rev_fixed_b": lambda: fixtures.random_chain(626, 8, p_prismatic=0.0, p_fixed=0.3)}
CHAINS = ["c6", "c7", "c6_perturbed", "rev_fixed_a", "rev_fixed_b"]


def _desc(name):
    return RANDOM[name]() if name in RANDOM else fixtures.by_name(name)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


def _inputs(torch, n_in, n, seed):
    rng = np.random.RandomState(seed)
    q, dq, ddq = rng.uniform(-np.pi, np.pi, (n_in, n)), rng.uniform(-2, 2, (n_in, n)), rng.uniform(-5, 5, (n_in, n))
    return [torch.tensor(x, device="cuda") for x in (q, dq, ddq)]


def _both(ch, fn, monkeypatch):
    """fn() with the specialised kernel, then with the precompiled one; returns both results (numpy) and the two kernel infos"""
    monkeypatch.delenv("RDB_GRAM_JIT", raising=False)
    a = [x.cpu().numpy().copy() for x in fn()]
    ia = ch.gramKernelInfo()
    monkeypatch.setenv("RDB_GRAM_JIT", "0")
    b = [x.cpu().numpy().copy() for x in fn()]
    ib = ch.gramKernelInfo()
    monkeypatch.delenv("RDB_GRAM_JIT")
    return a, b, ia, ib


@pytest.mark.gpu
@pytest.mark.parametrize("name", CHAINS)
@pytest.mark.parametrize("n", [4096 * 37 + 13, 31])
def test_specialised_equals_precompiled(name, n, torch, monkeypatch):
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch = Chain(d)
    assert ch.gramKernelInfo()[0] == -1
    q, dq, ddq = _inputs(torch, d.n_inputs, n, 17 + n % 5)
    tau = torch.tensor(np.random.RandomState(3).uniform(-50, 50, (d.n_inputs, n)), device="cuda")
    for tm in (None, tau):  # computed and measured torques
        a, b, ia, ib = _both(ch, lambda: ch.regressorGram(q, dq, ddq, tau_meas=tm), monkeypatch)
        assert ia[0] == 1, ia[1]
        assert "NVRTC" in ia[1]
        assert ib[0] == 0 and "RDB_GRAM_JIT=0" in ib[1]
        for x, y, what in zip(a, b, ("gram", "rhs", "tau_sq")):
            assert np.array_equal(x, y), (name, what, np.max(np.abs(x - y)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7", "rev_fixed_a"])
def test_specialised_extended_model(name, torch, monkeypatch):
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch = Chain(d)
    n_in = d.n_inputs
    tn = {1: "friction1", 2: "friction2", 3: "spring"}
    ch.setComponents([{"type": tn[1 + (k % 3)], "joint": k % n_in, "min_velocity": 0.05, "max_velocity": 0.7} for k in range(n_in + 2)])
    q, dq, ddq = _inputs(torch, n_in, 100_003, 5)
    a, b, ia, ib = _both(ch, lambda: ch.regressorGramExt(q, dq, ddq), monkeypatch)
    assert ia[0] == 1 and ib[0] == 0, (ia, ib)
    for x, y in zip(a, b):
        assert np.array_equal(x, y), np.max(np.abs(x - y))


NON_FINITE = [("q", 1, float("nan")), ("q", 3, float("inf")), ("dq", 4, float("inf")), ("dq", 0, float("nan")), ("ddq", 0, -float("inf")),
              ("ddq", 5, float("nan"))]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7"])
@pytest.mark.parametrize("plane,joint,value", NON_FINITE)
def test_non_finite_input(name, plane, joint, value, torch, monkeypatch):
    """One non-finite input of one sample (computed torques).  The specialised kernel does not form 0 * inf or 0 * NaN with the exact zeros of
    the model, so it can leave a finite or differently non-finite value where the precompiled kernel has NaN.  What holds: wherever the
    precompiled result is finite, the specialised result is bit-identical (a finite result has only finite operands, and the specialised
    kernel computes the same operations minus products with exact 0 and +-1), and the sample does not vanish from either result."""
    from rosdyn_b200.chain import Chain
    d = fixtures.by_name(name)
    ch = Chain(d)
    n = 4096
    x = dict(zip(("q", "dq", "ddq"), _inputs(torch, d.n_inputs, n, 23)))
    x[plane][joint, 1234] = value
    a, b, ia, ib = _both(ch, lambda: ch.regressorGram(x["q"], x["dq"], x["ddq"]), monkeypatch)
    assert ia[0] == 1 and ib[0] == 0
    for spec, pre in zip(a, b):
        fin = np.isfinite(pre)
        assert np.array_equal(spec[fin], pre[fin])
        assert not fin.all() and not np.isfinite(spec).all()
    # the non-finite sample also poisons tau_sq in both
    assert not np.isfinite(a[2][0]) and not np.isfinite(b[2][0])


@pytest.mark.gpu
def test_generic_chain_reports_the_precompiled_kernel(torch):
    from rosdyn_b200.chain import Chain
    d = fixtures.random_chain(11, 6, p_prismatic=0.5, p_fixed=0.0)
    ch = Chain(d)
    q, dq, ddq = _inputs(torch, d.n_inputs, 1000, 1)
    ch.regressorGram(q, dq, ddq)
    torch.cuda.synchronize()
    flag, why = ch.gramKernelInfo()
    assert flag == 0 and "revolute" in why, why


_NO_NVRTC = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from rosdyn_b200 import fixtures
from rosdyn_b200.chain import Chain
d = fixtures.by_name("c6")
ch = Chain(d)
rng = np.random.RandomState(2)
q, dq, ddq = (torch.tensor(rng.uniform(-1, 1, (6, 5000)), device="cuda") for _ in range(3))
G = ch.regressorGram(q, dq, ddq)[0].cpu().numpy()
flag, why = ch.gramKernelInfo()
print(flag)
print(why)
np.save(sys.argv[2], G)
"""


@pytest.mark.gpu
def test_fallback_when_nvrtc_cannot_be_loaded(tmp_path, torch):
    outs = {}
    for tag, extra in (("missing", {"RDB_NVRTC_LIB": "libnvrtc-not-installed.so.12"}), ("disabled", {"RDB_GRAM_JIT": "0"})):
        env = dict(os.environ, **extra)
        r = subprocess.run([sys.executable, "-c", _NO_NVRTC, ROOT, str(tmp_path / f"{tag}.npy")], env=env, capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0, r.stderr
        flag, why = r.stdout.strip().splitlines()[-2:]
        assert flag == "0", why
        outs[tag] = np.load(tmp_path / f"{tag}.npy")
        if tag == "missing":
            assert "NVRTC not found" in why, why
    assert np.array_equal(outs["missing"], outs["disabled"])
