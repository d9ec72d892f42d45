"""GPU tests of parameter generation (zk_groth16_generate / groth16.generate_parameters, bellman's generate_parameters): byte parity
with the closed-form CRS of synthetic.make_toy_crs (which shares no code with the kernels), non-standard generators, sampled points of
a 2^20-constraint circuit, generate -> prove -> verify end to end, the error cases, and determinism."""
import random

import numpy as np
import pytest

from oracle import coracle as co
from oracle import pyref as pr
from zero_chain_b200 import groth16 as zk
from zero_chain_b200 import synthetic as sy

pytestmark = pytest.mark.gpu
R = pr.R

SHAPES = {
    "tiny": dict(n_constraints=60, n_inputs=4, n_aux=50, a_aux_density=40, b_density=33),
    "mid": dict(n_constraints=1500, n_inputs=23, n_aux=1400, a_aux_density=1000, b_density=800),
    "conf": sy.CONF_SHAPE,
    "anon": sy.ANON_SHAPE,
}
G1 = co.g1_encode(co.g1_generator(), False)
G2 = co.g2_encode(co.g2_generator(), False)


@pytest.fixture(scope="module")
def ctx():
    c = zk.Context(0)
    yield c
    c.close()


def _cs(ctx, r1cs):
    return zk.ConstraintSystem(ctx, r1cs.n_inputs, r1cs.n_aux, r1cs.A, r1cs.B, r1cs.C)


def _gen(cs, td, g1=G1, g2=G2):
    return zk.generate_parameters(cs, g1, g2, td["alpha"], td["beta"], td["gamma"], td["delta"], td["tau"])


@pytest.mark.parametrize("shape", ["tiny", "mid", "conf", "anon"])
def test_generate_matches_closed_form_crs(ctx, shape):
    r1cs = sy.make_r1cs(seed=3, **SHAPES[shape])
    crs = sy.make_toy_crs(r1cs, co.g1_fixed_base, co.g2_fixed_base, seed=4)
    cs = _cs(ctx, r1cs)
    p = _gen(cs, crs.trapdoor)
    assert p.write() == crs.params_bytes
    cs.free(); p.free()


@pytest.mark.parametrize("shape", ["tiny", "mid"])
def test_generate_non_standard_generators(ctx, shape):
    r1cs = sy.make_r1cs(seed=5, **SHAPES[shape])
    b1 = co.g1_fixed_base(co.ints_to_limbs([0xC0FFEE1234], 4))[0]
    b2 = co.g2_fixed_base(co.ints_to_limbs([R - 77], 4))[0]
    crs = sy.make_toy_crs(r1cs, lambda s: co.g1_fixed_base(s, base=b1), lambda s: co.g2_fixed_base(s, base=b2), seed=6)
    cs = _cs(ctx, r1cs)
    p = _gen(cs, crs.trapdoor, co.g1_encode(b1, False), co.g2_encode(b2, False))
    assert p.write() == crs.params_bytes
    cs.free(); p.free()


def _qap(r1cs, tau, vars_):
    """at, bt, ct of the given variables from the column entries and the Lagrange coefficients at tau (python integers)."""
    n_rows = r1cs.n_constraints + r1cs.n_inputs
    log_m = max(1, (n_rows - 1).bit_length())
    m = 1 << log_m
    w = pow(sy._ROOT, 1 << (32 - log_m), R)
    zt = (pow(tau, m, R) - 1) % R
    k = zt * pow(m, -1, R) % R
    Lj = lambda j: k * pow(w, j, R) % R * pow((tau - pow(w, j, R)) % R, -1, R) % R
    want = set(vars_)
    out = {v: [0, 0, 0] for v in want}
    for mi, M in enumerate((r1cs.A, r1cs.B, r1cs.C)):
        for j, row in enumerate(M):
            hit = [(v, c) for v, c in row if v in want]
            if hit:
                l = Lj(j)
                for v, c in hit:
                    out[v][mi] = (out[v][mi] + c * l) % R
    for v in want:
        if v < r1cs.n_inputs:
            out[v][0] = (out[v][0] + Lj(r1cs.n_constraints + v)) % R
    return out, zt, m


def test_generate_scale_2p20_sampled(ctx):
    """2^20 constraints (domain 2^21): 256 sampled points of every vector against k g with k computed in Python."""
    n = 1 << 20
    r1cs = sy.make_r1cs(n, 23, n - 64, (n - 64) * 4 // 5, (n - 64) * 5 // 8, seed=9)
    td = dict(tau=0x1234567 << 200, alpha=R - 5, beta=0xABCDEF << 100, gamma=0x77 << 220, delta=3 ** 150 % R)
    cs = _cs(ctx, r1cs)
    p = _gen(cs, td)
    buf = p.write()
    lay = {k: o for k, (o, _) in pr.params_layout(buf).items()}
    rng = random.Random(11)
    a_d, bi_d, ba_d = sy.densities(r1cs)
    n_in = r1cs.n_inputs
    a_vars = list(range(n_in)) + [n_in + i for i in np.flatnonzero(a_d)]
    b_vars = [i for i in np.flatnonzero(bi_d)] + [n_in + i for i in np.flatnonzero(ba_d)]
    assert (p.n_a, p.n_b_g1, p.n_l, p.n_h) == (len(a_vars), len(b_vars), r1cs.n_aux, (1 << 21) - 1)
    pick = {k: sorted(rng.sample(range(cnt), min(256, cnt))) for k, cnt in (("h", p.n_h), ("l", p.n_l), ("a", p.n_a), ("b", p.n_b_g1))}
    pick["ic"] = [3, n_in - 1]                   # ONE and inputs 1, 2 sit in most rows of B: left to the closed-form tests above
    need = {n_in + i for i in pick["l"]} | {a_vars[i] for i in pick["a"]} | {b_vars[i] for i in pick["b"]} | set(pick["ic"])
    q, zt, m = _qap(r1cs, td["tau"], need)
    ginv, dinv = pow(td["gamma"], -1, R), pow(td["delta"], -1, R)
    comb = lambda v: (td["beta"] * q[v][0] + td["alpha"] * q[v][1] + q[v][2]) % R
    checks = [("h", i, pow(td["tau"], i, R) * zt % R * dinv % R, 1) for i in pick["h"]]
    checks += [("l", i, comb(n_in + i) * dinv % R, 1) for i in pick["l"]]
    checks += [("a", i, q[a_vars[i]][0], 1) for i in pick["a"]]
    checks += [("b_g1", i, q[b_vars[i]][1], 1) for i in pick["b"]] + [("b_g2", i, q[b_vars[i]][1], 2) for i in pick["b"]]
    checks += [("ic", i, comb(i) * ginv % R, 1) for i in pick["ic"]]
    for grp in (1, 2):
        sel = [c for c in checks if c[3] == grp]
        want = (co.g1_fixed_base if grp == 1 else co.g2_fixed_base)(co.ints_to_limbs([c[2] for c in sel], 4), enc=True)
        sz = 96 * grp
        got = b"".join(buf[lay[c[0]] + sz * c[1]: lay[c[0]] + sz * (c[1] + 1)] for c in sel)
        assert got == bytes(want)
    cs.free(); p.free()


def test_generate_random_prove_verify(ctx):
    """generate_random_parameters -> proofs from witnesses equal the closed form -> accepted by the device verifier and by the
    oracle's, a tampered public input rejected by both; a checked read of the written bytes writes them back unchanged."""
    r1cs = sy.make_r1cs(seed=21, **SHAPES["mid"])
    cs = _cs(ctx, r1cs)
    p = zk.generate_random_parameters(cs, random.Random(2024))
    # the same draws as generate_random_parameters: k1, k2, then alpha, beta, gamma, delta, tau
    rr = random.Random(2024)
    k1, k2 = 1 + rr.randrange(R) % (R - 1), 1 + rr.randrange(R) % (R - 1)
    alpha, beta, gamma, delta, tau = (rr.randrange(R) for _ in range(5))
    q, zt, m = _qap(r1cs, tau, range(r1cs.n_inputs + r1cs.n_aux))
    nv = r1cs.n_inputs + r1cs.n_aux
    crs = sy.ToyCRS(b"", dict(tau=tau, alpha=alpha, beta=beta, gamma=gamma, delta=delta), [q[v][0] for v in range(nv)],
                    [q[v][1] for v in range(nv)], [q[v][2] for v in range(nv)], zt, m.bit_length() - 1, r1cs)
    batch = 2
    zs = [sy.make_witness(r1cs, 60 + k) for k in range(batch)]
    rs, ss = [0x1111, 0x2222], [0x3333, 0x4444]
    inputs = np.stack([co.ints_to_limbs(z[:r1cs.n_inputs], 4) for z in zs])
    aux = np.stack([co.ints_to_limbs(z[r1cs.n_inputs:], 4) for z in zs])
    proofs = zk.create_proof_from_witness_batch(cs, p, batch, inputs, aux, co.ints_to_limbs(rs, 4), co.ints_to_limbs(ss, 4))
    for k in range(batch):
        A, B, Cc = sy.expected_proof_scalars(crs, zs[k], rs[k], ss[k])
        want = pr.proof_bytes(pr.ec_mul(pr.FQ, pr.G1_GEN, A * k1 % R), pr.ec_mul(pr.FQ2, pr.G2_GEN, B * k2 % R), pr.ec_mul(pr.FQ, pr.G1_GEN, Cc * k1 % R))
        assert proofs[192 * k:192 * (k + 1)] == want, k
    pk, vk = zk.parameter_files(p)
    pvk = zk.PreparedVerifyingKey.prepare(ctx, p.vk_bytes())
    opvk = co.PreparedVerifyingKey.prepare(p.vk_bytes())
    assert pvk.write() == opvk.write() == vk
    ins = [zs[0][1:r1cs.n_inputs], zs[1][1:r1cs.n_inputs]]
    bad = [list(ins[0]), list(ins[1])]
    bad[1][0] = (bad[1][0] + 1) % R
    assert zk.verify_proofs(pvk, proofs, ins) == [1, 1]
    assert zk.verify_proofs(pvk, proofs, bad) == [1, 0]
    n_pub = r1cs.n_inputs - 1
    assert opvk.verify_batch(proofs, co.ints_to_limbs(ins[0] + ins[1], 4), n_pub) == [1, 1]
    assert opvk.verify_batch(proofs, co.ints_to_limbs(bad[0] + bad[1], 4), n_pub) == [1, 0]
    back = zk.Parameters.read(ctx, pk, checked=True)
    assert back.write() == pk
    back.free(); pvk.free(); cs.free(); p.free()


def _raises(code, fn):
    with pytest.raises(zk.SynthesisError) as e:
        fn()
    assert e.value.code == code, e.value


def test_generate_errors(ctx):
    r1cs = sy.make_r1cs(seed=3, **SHAPES["tiny"])
    cs = _cs(ctx, r1cs)
    td = dict(tau=5, alpha=6, beta=7, gamma=8, delta=9)
    gen = lambda **kw: _gen(cs, {**td, **kw}).free()
    for k in ("gamma", "delta", "alpha", "beta", "tau"):
        _raises(-5, lambda: gen(**{k: 0}))
    m = 64                                                             # 60 constraints + 4 inputs
    _raises(-5, lambda: gen(tau=pow(sy._ROOT, (1 << 32) // m, R)))     # primitive m-th root of unity: t(tau) = 0
    _raises(-8, lambda: gen(delta=R))
    # generators: off the curve, on the curve outside the r-torsion, at infinity
    off = bytearray(G1); off[95] ^= 1
    _raises(-7, lambda: _gen(cs, td, bytes(off)).free())
    off2 = bytearray(G2); off2[191] ^= 1
    _raises(-7, lambda: _gen(cs, td, G1, bytes(off2)).free())
    x = 4
    while True:
        y = pr.FQ.sqrt((x ** 3 + 4) % pr.Q)
        if y is not None and pr.ec_mul(pr.FQ, (x, y), R) is not pr.INF:
            break
        x += 1
    _raises(-7, lambda: _gen(cs, td, pr.g1_uncompressed((x, y))).free())
    _raises(-5, lambda: _gen(cs, td, bytes([0x40]) + bytes(95)).free())
    _raises(-5, lambda: _gen(cs, td, G1, bytes([0x40]) + bytes(191)).free())
    cs.free()
    # an aux variable used in no row: its l point is the identity
    un = sy.make_r1cs(seed=3, **SHAPES["tiny"])
    un.n_aux += 1
    cs2 = _cs(ctx, un)
    _raises(-10, lambda: _gen(cs2, td).free())
    cs2.free()


def test_generate_cancelling_b_column(ctx):
    """A B row holding c and r - c for one variable: bt = 0, so bellman drops its point from b_g1 and b_g2 by value; the same variable
    has an A entry, so its a point stays."""
    r1cs = sy.make_r1cs(seed=3, **SHAPES["tiny"])
    v = r1cs.n_inputs + r1cs.n_bool + 5
    for row in r1cs.B:
        row[:] = [(x, c) for x, c in row if x != v]
    r1cs.B[7] = r1cs.B[7] + [(v, 12345), (v, R - 12345)]
    r1cs.A[7] = r1cs.A[7] + [(v, 3)]
    crs = sy.make_toy_crs(r1cs, co.g1_fixed_base, co.g2_fixed_base, seed=4)     # filters by density: keeps v's identity in b
    assert crs.bt[v] == 0 and crs.at[v] != 0
    cs = _cs(ctx, r1cs)
    p = _gen(cs, crs.trapdoor)
    a_d, bi_d, ba_d = sy.densities(r1cs)
    b_vars = [int(i) for i in np.flatnonzero(bi_d)] + [r1cs.n_inputs + int(i) for i in np.flatnonzero(ba_d)]
    assert (p.n_a, p.n_b_g1, p.n_b_g2) == (r1cs.n_inputs + int(a_d.sum()), len(b_vars) - 1, len(b_vars) - 1)
    assert p.write() == _drop_point(crs.params_bytes, b_vars.index(v))
    cs.free(); p.free()


def _drop_point(buf, k):
    """Remove point k of b_g1 and of b_g2 from a Parameters stream (the two u32 counts decrease by one)."""
    import struct
    off = 96 + 96 + 192 + 192 + 96 + 192
    out = bytearray(buf[:off])
    for vec, sz in (("ic", 96), ("h", 96), ("l", 96), ("a", 96), ("b_g1", 96), ("b_g2", 192)):
        n = struct.unpack(">I", buf[off:off + 4])[0]
        body = buf[off + 4: off + 4 + n * sz]
        if vec in ("b_g1", "b_g2"):
            body = body[:k * sz] + body[(k + 1) * sz:]
            n -= 1
        out += struct.pack(">I", n) + body
        off += 4 + (n + (1 if vec in ("b_g1", "b_g2") else 0)) * sz
    return bytes(out)


def test_generate_deterministic_across_contexts(ctx):
    r1cs = sy.make_r1cs(seed=3, **SHAPES["mid"])
    td = dict(tau=11, alpha=12, beta=13, gamma=14, delta=15)
    c2 = zk.Context(0)
    outs = []
    for c in (ctx, c2):
        cs = _cs(c, r1cs)
        p = _gen(cs, td)
        outs.append(p.write())
        p.free(); cs.free()
    c2.close()
    assert outs[0] == outs[1]
