"""CPU check of parameter generation's per-thread device code (zero_chain_b200/csrc/setup.cuh) compiled with ZK_HOST_EMUL
(tests/host_emul/emul_setup.cpp): the signed-digit recoding of full 256-bit scalars, the fixed-base table walk against the oracle's
scalar multiplication, the affine conversion with one shared inverse (identities included), and the bounded segmented column
sums of the QAP evaluation against Python integers.  The device build of the same source is covered by tests/test_gpu_setup.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import coracle as co
from oracle import pyref as pr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SPECIAL = [0, 1, 2, pr.R - 1, pr.R, (1 << 255) - 1, 1 << 255, (1 << 256) - 1, 0x5555 << 240, (1 << 256) - (1 << 128)]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emuls") / "libemuls.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "zero_chain_b200", "csrc"),
                           "-o", so, os.path.join(HERE, "host_emul", "emul_setup.cpp")])
    return C.CDLL(so)


def _u256(rng):
    return sum(rng.next() << (64 * i) for i in range(4))


def _words(ks):
    return np.array([[(k >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for k in ks], np.uint32)


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("c", [6, 8, 10, 12])
def test_signed_digit_recoding(emu, c):
    rng = pr.SplitMix64(c)
    W = emu.emu_windows(c)
    assert W == 256 // c + 1
    for k in SPECIAL + [_u256(rng) for _ in range(300)]:
        d = np.zeros(W, np.int32)
        assert emu.emu_recode(_vp(_words([k])), c, _vp(d)) == 0                      # no carry left over
        assert all(-(1 << (c - 1)) < int(x) <= 1 << (c - 1) for x in d)
        assert sum(int(x) << (c * w) for w, x in enumerate(d)) == k


@pytest.mark.parametrize("g,c", [(1, 6), (1, 8), (1, 10), (1, 12), (2, 6), (2, 12)])
def test_table_walk_matches_oracle(emu, g, c):
    """k g through the table for full 256-bit k (reduced mod r by the group), at a non-standard generator."""
    rng = pr.SplitMix64(100 + c)
    ks = SPECIAL + [_u256(rng) for _ in range(12)]
    fixed, mul, w = (co.g1_fixed_base, co.g1_mul, 12) if g == 1 else (co.g2_fixed_base, co.g2_mul, 24)
    base = np.ascontiguousarray(fixed(co.ints_to_limbs([0x1234567], 4))[0])
    out = np.zeros((len(ks), w), np.uint64)
    getattr(emu, "emu_g%d_walk" % g)(_vp(base), _vp(_words(ks)), len(ks), c, _vp(out))
    for i, k in enumerate(ks):
        assert np.array_equal(out[i], mul(base, k % pr.R)), (i, hex(k))


@pytest.mark.parametrize("g", [1, 2])
def test_shared_inverse_normalisation(emu, g):
    """A batch with identities in it (first, middle, last): every point equals the oracle's 2 P, identities stay all-zero."""
    fixed, dbl, w = (co.g1_fixed_base, co.g1_double, 12) if g == 1 else (co.g2_fixed_base, co.g2_double, 24)
    ks = [0, 3, 5, 0, 7, pr.R - 1, 11, 0, 13, 2, 0]
    pts = np.ascontiguousarray(fixed(co.ints_to_limbs(ks, 4)))
    out = np.zeros_like(pts)
    getattr(emu, "emu_g%d_normalize" % g)(_vp(pts), len(ks), _vp(out))
    for i in range(len(ks)):
        assert np.array_equal(out[i], dbl(pts[i])), i
    assert not out[0].any() and not out[-1].any()


@pytest.mark.parametrize("nnz,nv,heavy", [(0, 5, 0), (1, 3, 0), (31, 4, 0), (33, 2, 1), (5000, 300, 2000), (40000, 10, 39000)])
def test_segmented_column_sums(emu, nnz, nv, heavy):
    """Columns of every length, one column carrying `heavy` entries (the ONE variable in the boolean rows of B), empty columns."""
    rng = pr.SplitMix64(nnz + nv)
    cols = [0] * heavy + [rng.next() % nv for _ in range(nnz - heavy)]
    vals = [rng.fr() for _ in range(nnz)]
    out = np.zeros((nv, 8), np.uint32)
    col = np.array(cols or [0], np.uint32)
    v = _words(vals) if nnz else np.zeros((1, 8), np.uint32)
    passes = emu.emu_column_sums(_vp(col), _vp(v), C.c_size_t(nnz), C.c_size_t(nv), _vp(out))
    want = [0] * nv
    for cc, x in zip(cols, vals):
        want[cc] = (want[cc] + x) % pr.R
    got = [sum(int(x) << (32 * i) for i, x in enumerate(row)) for row in out]
    assert got == want                         # Montgomery form is additive: the sums compare as plain residues
    assert passes == (0 if nnz <= 1 else int(np.ceil(np.log(nnz) / np.log(32) - 1e-9)))
