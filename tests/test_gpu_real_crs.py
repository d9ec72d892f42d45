"""GPU parity tests on a sample of the reference's SHIPPED proving key (zface/params/conf_pk.dat: its vk and the first points of
every query, committed as tests/golden/conf_pk_sample.dat by tests/golden/make_golden.py): the call the device loader replaces
is `Parameters::read(&pk_buf[..], true)` at core/proofs/src/confidential.rs:95-103, the writer `self.proving_key.write(..)` at
confidential.rs:73-93.

Every toy CRS in the other tests consists of known multiples of the generator made by this repo's own code; the 2 952 points of
the sample are not, so a decoding or group-law defect that only "foreign" points trigger shows up here.  A real
confidential_transfer witness cannot be made here (it needs the Rust gadget library), so the proofs use a synthetic assignment of
the sample's shape — they do not verify under conf_vk.dat, but their bytes must equal the oracle's on the same CRS and inputs."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import coracle as co
from oracle import pyref as pr
from zero_chain_b200 import groth16 as zk
from zero_chain_b200 import synthetic as sy

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
COUNTS = (23, 1023, 623, 509, 387, 387)                   # ic, h, l, a, b_g1, b_g2 of the sample (about 1/32 of every query)
# the circuit the sample is the proving key of: domain 2^10, a = inputs + a_aux_density, b = b_density
SHAPE = dict(n_constraints=624, n_inputs=23, n_aux=623, a_aux_density=486, b_density=387)


@pytest.fixture(scope="module")
def ctx():
    c = zk.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def pk():
    buf = open(os.path.join(GOLD, "conf_pk_sample.dat"), "rb").read()
    S = json.load(open(os.path.join(GOLD, "kats.json")))["conf_pk_sample"]
    assert len(buf) == S["size"] and hashlib.sha256(buf).hexdigest() == S["sha256"]
    return buf


@pytest.fixture(scope="module")
def params(ctx, pk):
    p = zk.Parameters.read(ctx, pk, checked=True)          # on-curve + r-torsion tests of every point on the device
    yield p
    p.free()


def _assignment(seed):
    """A synthetic ProvingAssignment of the sample's shape: c = a * b on every row (so that H is a polynomial),
    ~90 % of the aux values in {0, 1} like a boolean-heavy witness, densities with the sample's counts."""
    sh = SHAPE
    n_in, n_aux = sh["n_inputs"], sh["n_aux"]
    n_c = sh["n_constraints"] + n_in
    rng = sy.SplitMix64(seed)
    a = [rng.fr() for _ in range(n_c)]
    b = [rng.fr() for _ in range(n_c)]
    c = [x * y % pr.R for x, y in zip(a, b)]
    aux = [(rng.next() & 1) if rng.next() % 10 else rng.fr() for _ in range(n_aux)]
    inputs = [1] + [rng.fr() for _ in range(n_in - 1)]
    a_d = np.zeros(n_aux, np.uint8); a_d[np.random.RandomState(seed).permutation(n_aux)[:sh["a_aux_density"]]] = 1
    b_in = np.zeros(n_in, np.uint8); b_in[:2] = 1
    b_d = np.zeros(n_aux, np.uint8); b_d[np.random.RandomState(seed + 1).permutation(n_aux)[:sh["b_density"] - 2]] = 1
    L = lambda v: co.ints_to_limbs(v, 4)
    return zk.ProvingAssignment(L(a), L(b), L(c), L(inputs), L(aux), a_d, b_in, b_d)


def _oracle_prove(op, pa, r, s):
    return op.prove(pa.a, pa.b, pa.c, pa.input_assignment, pa.aux_assignment, pa.a_aux_density, pa.b_input_density, pa.b_aux_density, r, s)


def test_shipped_crs_loads_checked_and_round_trips(ctx, pk, params):
    assert (params.n_ic, params.n_h, params.n_l, params.n_a, params.n_b_g1, params.n_b_g2) == COUNTS
    # Parameters::write of the resident CRS reproduces the sample byte for byte (decode -> Montgomery -> encode)
    out = params.write()
    assert len(out) == len(pk) and hashlib.sha256(out).digest() == hashlib.sha256(pk).digest() and out == pk
    # params.vk (setup.rs:31) and prepare_verifying_key of it = the shipped conf_vk.dat
    head = open(os.path.join(GOLD, "conf_vk_head.bin"), "rb").read()
    assert params.vk_bytes() == head == pk[:len(head)]
    pvk = zk.PreparedVerifyingKey.prepare(ctx, params.vk_bytes())
    assert pvk.write() == open(os.path.join(GOLD, "conf_pvk.dat"), "rb").read()
    pvk.free()


def test_proofs_on_the_shipped_crs_equal_the_oracle(ctx, pk, params):
    op = co.Params(pk, checked=False)
    assert (op.n_ic, op.n_h, op.n_l, op.n_a, op.n_b) == COUNTS[:5]
    rng = pr.SplitMix64(2024)
    pas, rs, ss = [], [], []
    for seed in (1, 2, 3):
        pas.append(_assignment(seed)); rs.append(rng.fr()); ss.append(rng.fr())
    want = [_oracle_prove(op, pa, r, s) for pa, r, s in zip(pas, rs, ss)]
    assert zk.create_proof(pas[0], params, rs[0], ss[0]) == want[0]
    # densities are per circuit: a batch shares them, so the batch uses one assignment shape with three value sets
    same = [pas[0]]
    for k in (1, 2):
        q = _assignment(k + 1)
        same.append(zk.ProvingAssignment(q.a, q.b, q.c, q.input_assignment, q.aux_assignment, pas[0].a_aux_density, pas[0].b_input_density, pas[0].b_aux_density))
    got = zk.create_proof_batch(same, params, rs, ss)
    for k in range(3):
        assert got[192 * k:192 * (k + 1)] == _oracle_prove(op, same[k], rs[k], ss[k]), k
    # the proofs are well-formed group elements (Proof::read accepts them); they cannot verify: the witness is synthetic
    for k in range(3):
        pr.proof_read(got[192 * k:192 * (k + 1)])


def test_corrupted_shipped_crs_is_rejected(ctx, pk):
    lay = pr.params_layout(pk)
    off = lay["a"][0] + 96 * (lay["a"][1] * 3 // 4)
    bad = bytearray(pk); bad[off + 95] ^= 1                                   # y changed: not on the curve
    with pytest.raises(zk.SynthesisError) as e:
        zk.Parameters.read(ctx, bytes(bad), checked=True)
    assert e.value.code == -7
    zk.Parameters.read(ctx, bytes(bad), checked=False).free()                 # unchecked read accepts any field elements (bellman)
    # a point on the curve but outside the r-torsion, in the h query
    x = 0
    while True:
        y = pr.FQ.sqrt((x ** 3 + 4) % pr.Q)
        if y is not None and pr.ec_mul(pr.FQ, (x, y), pr.R) is not pr.INF:
            break
        x += 1
    off = lay["h"][0] + 96 * (lay["h"][1] - 30)
    bad = bytearray(pk); bad[off:off + 96] = x.to_bytes(48, "big") + y.to_bytes(48, "big")
    with pytest.raises(zk.SynthesisError) as e:
        zk.Parameters.read(ctx, bytes(bad), checked=True)
    assert e.value.code == -7
    # (0, 0) without the infinity flag is NotOnCurve in the reference (ec.rs:675-685), never the point at infinity
    off = lay["ic"][0] + 96 * 3
    bad = bytearray(pk); bad[off:off + 96] = bytes(96)
    with pytest.raises(zk.SynthesisError) as e:
        zk.Parameters.read(ctx, bytes(bad), checked=True)
    assert e.value.code == -7
    with pytest.raises(zk.SynthesisError):
        zk.Parameters.read(ctx, pk[:-5], checked=True)                        # truncated stream


def test_decoded_crs_cache(ctx, pk, params, tmp_path):
    path = str(tmp_path / "conf_pk.zkcache")
    pa = _assignment(7)
    want = zk.create_proof(pa, params, 11, 22)
    p1 = zk.Parameters.read_cached(ctx, pk, path)
    assert not p1.cache_hit and os.path.getsize(path) > 0.9 * len(pk)
    p2 = zk.Parameters.read_cached(ctx, pk, path)
    assert p2.cache_hit
    for p in (p1, p2):
        assert zk.create_proof(pa, p, 11, 22) == want and p.write() == pk
        p.free()
    # another key (one byte changed, still a valid stream prefix-wise) must miss — and fail the checked load
    other = bytearray(pk); other[pr.params_layout(pk)["l"][0] + 95] ^= 1
    with pytest.raises(zk.SynthesisError):
        zk.Parameters.read_cached(ctx, bytes(other), path)
    # a cache whose BODY was altered (header intact) must not be trusted: it is ignored and rewritten
    with open(path, "r+b") as f:
        f.seek(len(pk) // 2); b = f.read(1); f.seek(len(pk) // 2); f.write(bytes([b[0] ^ 1]))
    p4 = zk.Parameters.read_cached(ctx, pk, path)
    assert not p4.cache_hit and zk.create_proof(pa, p4, 11, 22) == want
    p4.free()
    assert zk.Parameters.read_cached(ctx, pk, path).cache_hit
    # a truncated cache file is ignored and rewritten
    open(path, "r+b").truncate(len(pk) // 10)
    p3 = zk.Parameters.read_cached(ctx, pk, path)
    assert not p3.cache_hit and os.path.getsize(path) > 0.9 * len(pk)
    p3.free()
