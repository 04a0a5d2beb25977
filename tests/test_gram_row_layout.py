"""Row layout of the fused normal-equation kernel on all-revolute chains (GramGeom Z = 2, csrc/gram_common.cuh), without a GPU.

The kernel stores, per row of the folded regressor, only the columns that are not exact zeros of the all-revolute walk: on its own joint a link
has no m and no m c_z term, and the first moving link (on the fixed base) keeps only I_zz, m c_x and m c_y.  Here the layout the library
reports (rdb_gram_row_layout) is checked to cover every other (row, column) exactly once, and every column it drops is checked to be an exact
zero (to the rounding of the oracle's general formulas) of the oracle's regressor in the canonical frames of the folded chain, for random
samples."""
import ctypes

import numpy as np
import pytest

from rosdyn_b200.descriptor import REVOLUTE
from test_canonical_frames import RANDOM, _canonical, _desc

M, MCX, MCY, MCZ, IZZ = 0, 1, 2, 3, 9


def _layout(nj):
    from rosdyn_b200._lib import load
    pos, rowlen, tc = np.zeros(10 * nj * nj, dtype=np.int32), np.zeros(nj, dtype=np.int32), ctypes.c_int32(-1)
    p32 = ctypes.POINTER(ctypes.c_int32)
    assert load().rdb_gram_row_layout(nj, pos.ctypes.data_as(p32), rowlen.ctypes.data_as(p32), ctypes.byref(tc)) == 0
    return pos.reshape(nj, 10 * nj), rowlen, tc.value


def test_invalid_joint_counts_are_refused():
    from rosdyn_b200._lib import load
    p32 = ctypes.POINTER(ctypes.c_int32)
    buf, tc = np.zeros(1000, dtype=np.int32), ctypes.c_int32()
    for nj in (0, 8, -1):
        assert load().rdb_gram_row_layout(nj, buf.ctypes.data_as(p32), buf.ctypes.data_as(p32), ctypes.byref(tc)) != 0


@pytest.mark.parametrize("nj", range(1, 8))
def test_layout_covers_every_kept_entry_once(nj):
    pos, rowlen, tc = _layout(nj)
    assert tc in (0, 1)
    col_pos = {}
    for j in range(nj):
        kept = [c for c in range(10 * nj) if pos[j, c] >= 0]
        # a row holds the blocks of the links >= j, without the exact zeros of its own block (and of link 0 altogether)
        assert all(c // 10 >= j for c in kept)
        own = {c % 10 for c in kept if c // 10 == j}
        assert own == ({MCX, MCY, IZZ} if j == 0 else set(range(10)) - {M, MCZ}), (j, own)
        assert len(kept) == 10 * (nj - 1 - j) + len(own)
        # a dense prefix of positions behind tau, each used once
        assert sorted(pos[j, kept]) == list(range(tc, rowlen[j])), j
        for c in kept:  # a column sits at the same position in every row that holds it
            assert col_pos.setdefault(c, pos[j, c]) == pos[j, c]
    # the kernel's row 0 is its longest: tile count and DMMA count follow from the row lengths
    assert rowlen[0] == max(rowlen)
    if nj == 6:
        assert list(rowlen) == ([53, 48, 38, 28, 18, 8] if tc == 0 else [54, 49, 39, 29, 19, 9])
    if nj == 7:
        assert list(rowlen) == ([63, 58, 48, 38, 28, 18, 8] if tc == 0 else [64, 59, 49, 39, 29, 19, 9])


def _dmma_per_4_samples(rowlen):
    """row j needs the upper-triangular tiles among its tj(j) = ceil(rowlen / 8) tile columns"""
    return sum(t * (t + 1) // 2 for t in ((r + 7) // 8 for r in rowlen))


def test_dmma_counts_of_the_c6_and_c7_layouts():
    for nj, tiles_col, tiles_tau in ((6, 81, 90), (7, 125, 134)):
        _, rowlen, tc = _layout(nj)
        assert _dmma_per_4_samples(rowlen) == (tiles_col if tc == 0 else tiles_tau)


@pytest.mark.parametrize("name", ["c6", "c7", "c6_perturbed"] + list(RANDOM))
def test_dropped_columns_are_exact_zeros_of_the_folded_regressor(name):
    """Phi' of the chain in canonical frames (the frames of the folded chain; a moving link's block does not change when the links behind
    fixed joints are lumped into it): in the row of every moving joint, every column of a moving link that the layout drops is 0."""
    from oracle.oracle import OracleChain
    d = _desc(name)
    dc, _ = _canonical(d)
    moving = [k for k, jd in enumerate(d.joints) if jd.type == REVOLUTE]
    assert all(jd.type == REVOLUTE or jd.input_index < 0 for jd in d.joints)
    nj = len(moving)
    pos, _, _ = _layout(nj)
    rng = np.random.RandomState(11)
    n = 256
    q, dq, ddq = (rng.uniform(-np.pi, np.pi, (d.n_inputs, n)) for _ in range(3))
    phi, _ = OracleChain(dc).regressor_torque(q, dq, ddq)
    phi = phi.reshape(10 * d.n_joints, d.n_inputs, n)  # [column][input row][sample]
    scale = np.max(np.abs(phi), axis=(0, 2))  # per row
    dropped = kept_nonzero = 0
    worst = 0.0
    for j, kj in enumerate(moving):
        row = d.joints[kj].input_index
        for l, kl in enumerate(moving):
            if l < j:
                continue
            for p in range(10):
                v = phi[10 * kl + p, row]
                if pos[j, 10 * l + p] < 0:
                    worst = max(worst, np.max(np.abs(v)) / scale[row])
                    dropped += 1
                elif np.any(v != 0.0):
                    kept_nonzero += 1
    assert dropped == 7 + 2 * (nj - 1)
    # the kernel's walk produces these as exact zeros (typed Zr, or products of exact zeros); the oracle follows the reference's general
    # formulas, which leave rounding residue of a few ulps of the row's magnitude in some of them
    assert worst <= 1e-14, f"{name}: largest dropped entry {worst:.2e} of the row's magnitude"
    assert kept_nonzero > 0


# ---------------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c6", "c7", "c6_perturbed", "rev_fixed_a"])
@pytest.mark.parametrize("n", [4096 * 9 + 13, 31])
def test_gram_with_the_dropped_columns_against_oracle(name, n, torch):
    """G, b (accumulated beside the tiles) and tau^T tau against the oracle, odd batch tails, bit-reproducible, accumulate adds exactly."""
    from oracle.oracle import OracleChain
    from rosdyn_b200.chain import Chain
    d = _desc(name)
    ch, oc = Chain(d), OracleChain(d)
    rng = np.random.RandomState(n % 7)
    hq, hdq, hddq = rng.uniform(-np.pi, np.pi, (d.n_inputs, n)), rng.uniform(-2, 2, (d.n_inputs, n)), rng.uniform(-5, 5, (d.n_inputs, n))
    q, dq, ddq = (torch.tensor(x, device="cuda") for x in (hq, hdq, hddq))
    G, b, tt = (x.cpu().numpy() for x in ch.regressorGram(q, dq, ddq))
    assert ch.gramKernelInfo()[0] == 1
    Gr, br, tr = oc.gram(hq, hdq, hddq)
    assert np.max(np.abs(G - Gr)) <= 1e-10 * np.max(np.abs(Gr))
    assert np.max(np.abs(b - br)) <= 1e-10 * np.max(np.abs(br))
    assert abs(tt[0] - np.ravel(tr)[0]) <= 1e-10 * abs(np.ravel(tr)[0])
    again = [x.cpu().numpy() for x in ch.regressorGram(q, dq, ddq)]
    for x, y in zip((G, b, tt), again):
        assert np.array_equal(x, y)
    out = [torch.tensor(x, device="cuda") for x in (G, b, tt)]
    ch.regressorGram(q, dq, ddq, out=out)
    for x, y in zip((G, b, tt), out):
        assert np.array_equal(2 * x, y.cpu().numpy())
