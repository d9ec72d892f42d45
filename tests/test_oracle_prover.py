"""Checks the oracle's restatement of the UN-VENDORED bellman algorithms (multiexp, EvaluationDomain,
create_proof; SURVEY.md §3.2) against independent closed forms in Python big integers.  The
reference pins none of these outputs ("parity unpinned", SURVEY.md §8c), so these closed forms —
which share no code with the C oracle or the CUDA kernels — are the anchor."""
import numpy as np
import pytest

from oracle import coracle as co
from oracle import pyref as pr
from zero_chain_b200 import synthetic as sy


def _g1_ints(p):
    if not np.any(p):
        return pr.INF
    x, y = co.limbs_to_ints(np.asarray(p).reshape(2, 6))
    return (pr.fq_from_mont(x), pr.fq_from_mont(y))


def _g2_ints(p):
    if not np.any(p):
        return pr.INF
    v = [pr.fq_from_mont(x) for x in co.limbs_to_ints(np.asarray(p).reshape(4, 6))]
    return ((v[0], v[1]), (v[2], v[3]))


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 500, 4096])
def test_msm_g1_closed_form(n):
    # bases P_i = (i+1)*G as in the reference's vector files => MSM = (sum s_i (i+1)) * G
    rng = pr.SplitMix64(100 + n)
    bases = co.g1_fixed_base(co.ints_to_limbs(list(range(1, n + 1)), 4))
    scal = [rng.fr() for _ in range(n)]
    for k in range(0, n, 5):
        scal[k] = [0, 1, pr.R - 1, 2, 1][(k // 5) % 5]        # 0 / 1 fast paths and edge scalars
    got = co.g1_msm(bases, co.ints_to_limbs(scal, 4))
    k = sum(s * (i + 1) for i, s in enumerate(scal)) % pr.R
    assert _g1_ints(got) == pr.ec_mul(pr.FQ, pr.G1_GEN, k)


def test_msm_density_and_g2():
    n = 200
    rng = pr.SplitMix64(9)
    dens = np.array([rng.next() % 3 != 0 for _ in range(n)], np.uint8)
    nb = int(dens.sum())
    scal = [rng.fr() if rng.next() % 2 else rng.next() % 2 for _ in range(n)]
    b1 = co.g1_fixed_base(co.ints_to_limbs(list(range(1, nb + 1)), 4))
    b2 = co.g2_fixed_base(co.ints_to_limbs(list(range(1, nb + 1)), 4))
    k, j = 0, 0
    for i in range(n):
        if dens[i]:
            j += 1
            k += scal[i] * j
    k %= pr.R
    assert _g1_ints(co.g1_msm(b1, co.ints_to_limbs(scal, 4), dens)) == pr.ec_mul(pr.FQ, pr.G1_GEN, k)
    assert _g2_ints(co.g2_msm(b2, co.ints_to_limbs(scal, 4), dens)) == pr.ec_mul(pr.FQ2, pr.G2_GEN, k)
    # cancellation to infinity and repeated bases (exceptional cases of the mixed add)
    b = co.g1_fixed_base(co.ints_to_limbs([5, 5, 5, 5], 4))
    assert not np.any(co.g1_msm(b, co.ints_to_limbs([3, pr.R - 3, 7, pr.R - 7], 4)))
    assert _g1_ints(co.g1_msm(b, co.ints_to_limbs([9, 9, 9, 9], 4))) == pr.ec_mul(pr.FQ, pr.G1_GEN, 180)


def test_msm_rejects_identity_base():
    b = co.g1_fixed_base(co.ints_to_limbs([5, 0], 4))
    with pytest.raises(ValueError):
        co.g1_msm(b, co.ints_to_limbs([3, 4], 4))            # SynthesisError::UnexpectedIdentity


@pytest.mark.parametrize("log_n", [0, 1, 2, 5, 8])
def test_ntt_vs_bigint(log_n):
    n = 1 << log_n
    rng = pr.SplitMix64(log_n)
    x = [rng.fr() for _ in range(n)]
    xm = co.fr_to_mont(co.ints_to_limbs(x, 4))
    back = lambda a: co.limbs_to_ints(co.fr_from_mont(a))
    assert back(co.fr_ntt(xm, log_n, co.NTT_FFT)) == pr.ntt(x, log_n)
    assert back(co.fr_ntt(xm, log_n, co.NTT_IFFT)) == pr.intt(x, log_n)
    g = pr.FR_GENERATOR
    assert back(co.fr_ntt(xm, log_n, co.NTT_COSET_FFT)) == pr.ntt([v * pow(g, i, pr.R) % pr.R for i, v in enumerate(x)], log_n)
    gi = pow(g, -1, pr.R)
    assert back(co.fr_ntt(xm, log_n, co.NTT_ICOSET_FFT)) == [v * pow(gi, i, pr.R) % pr.R for i, v in enumerate(pr.intt(x, log_n))]
    # definition: out[k] = sum_j x[j] w^(jk)  (Horner at w^k)
    w = pr.omega(log_n)
    f = pr.ntt(x, log_n)
    for k in {0, n // 2, n - 1}:
        assert f[k] == pr.poly_eval(x, pow(w, k, pr.R))


def test_ntt_large_roundtrip_and_horner():
    log_n = 14
    n = 1 << log_n
    x = sy.random_fr_limbs(n, 3)
    xm = co.fr_to_mont(x)
    f = co.fr_ntt(xm, log_n, co.NTT_FFT)
    assert np.array_equal(co.fr_ntt(f, log_n, co.NTT_IFFT), xm)
    assert np.array_equal(co.fr_ntt(co.fr_ntt(xm, log_n, co.NTT_COSET_FFT), log_n, co.NTT_ICOSET_FFT), xm)
    xi = co.limbs_to_ints(x)
    fi = co.limbs_to_ints(co.fr_from_mont(f))
    w = pr.omega(log_n)
    for k in (1, 777, n - 1):
        assert fi[k] == pr.poly_eval(xi, pow(w, k, pr.R))


def _toy(shape, seed):
    r = sy.make_r1cs(seed=seed, **shape)
    crs = sy.make_toy_crs(r, co.g1_fixed_base, co.g2_fixed_base, seed=seed + 1)
    return r, crs


SMALL = dict(n_constraints=60, n_inputs=4, n_aux=50, a_aux_density=40, b_density=33)


def test_h_coeffs_vs_bigint():
    r = sy.make_r1cs(seed=2, **SMALL)
    z = sy.make_witness(r, 2)
    a, b, c = sy.evaluate(r, z)
    want = pr.h_coeffs(a, b, c, 6)
    got = co.limbs_to_ints(co.h_coeffs(co.ints_to_limbs(a, 4), co.ints_to_limbs(b, 4), co.ints_to_limbs(c, 4)))
    assert got == want
    # h * t == a*b - c as polynomials, evaluated at a random point
    x = 0x1234567
    n = 64
    ev = lambda evs: pr.poly_eval(pr.intt(list(evs) + [0] * (n - len(evs)), 6), x)
    assert pr.poly_eval(want, x) * (pow(x, n, pr.R) - 1) % pr.R == (ev(a) * ev(b) - ev(c)) % pr.R


@pytest.mark.parametrize("shape,seed", [(SMALL, 1), (SMALL, 2),
                                        (dict(n_constraints=300, n_inputs=23, n_aux=280, a_aux_density=200, b_density=150), 3)])
def test_create_proof_closed_form(shape, seed):
    r, crs = _toy(shape, seed)
    lay = pr.params_layout(crs.params_bytes)
    assert lay["end"][0] == len(crs.params_bytes)
    P = co.Params(crs.params_bytes, checked=True)
    a_d, bi_d, ba_d = sy.densities(r)
    assert P.n_a == r.n_inputs + int(a_d.sum()) and P.n_b == int(bi_d.sum() + ba_d.sum())
    z = sy.make_witness(r, seed)
    a, b, c = sy.evaluate(r, z)
    rng = pr.SplitMix64(seed + 77)
    rr, ss = rng.fr(), rng.fr()
    proof = P.prove(co.ints_to_limbs(a, 4), co.ints_to_limbs(b, 4), co.ints_to_limbs(c, 4),
                    co.ints_to_limbs(z[:r.n_inputs], 4), co.ints_to_limbs(z[r.n_inputs:], 4), a_d, bi_d, ba_d, rr, ss)
    A, B, C = sy.expected_proof_scalars(crs, z, rr, ss)
    want = pr.proof_bytes(pr.ec_mul(pr.FQ, pr.G1_GEN, A), pr.ec_mul(pr.FQ2, pr.G2_GEN, B), pr.ec_mul(pr.FQ, pr.G1_GEN, C))
    assert proof == want


def test_params_read_errors():
    r, crs = _toy(SMALL, 5)
    buf = bytearray(crs.params_bytes)
    with pytest.raises(ValueError):
        co.Params(bytes(buf[:-7]))                      # truncated
    lay = pr.params_layout(bytes(buf))
    off = lay["l"][0]
    bad = bytearray(buf); bad[off + 95] ^= 1            # corrupt a point
    co.Params(bytes(bad), checked=False)                # unchecked read accepts any field elements
    with pytest.raises(ValueError):
        co.Params(bytes(bad), checked=True)
    bad = bytearray(buf); bad[off:off + 96] = bytes([0x40]) + bytes(95)   # infinity in a query is rejected
    with pytest.raises(ValueError):
        co.Params(bytes(bad), checked=False)


def test_shipped_crs_parses():
    """Parameters grammar vs a sample of the reference's shipped CRS (tests/golden/conf_pk_sample.dat: the vk of
    zface/params/conf_pk.dat and the first points of every query, written by tests/golden/make_golden.py with the query
    lengths of the whole file).  SURVEY.md §3.3: the grammar must consume all bytes."""
    import hashlib, json, os
    gold = os.path.join(os.path.dirname(__file__), "golden")
    buf = open(os.path.join(gold, "conf_pk_sample.dat"), "rb").read()
    S = json.load(open(os.path.join(gold, "kats.json")))["conf_pk_sample"]
    assert hashlib.sha256(buf).hexdigest() == S["sha256"]
    assert buf.startswith(open(os.path.join(gold, "conf_vk_head.bin"), "rb").read())
    lay = pr.params_layout(buf)
    assert lay["end"][0] == len(buf) == S["size"]
    P = co.Params(buf, checked=True)          # on-curve + r-torsion for every point of the sample
    assert (P.n_ic, P.n_h, P.n_l, P.n_a, P.n_b) == (23,) + tuple(S["counts"][q] for q in ("h", "l", "a", "b_g1"))
    # the query lengths of the whole shipped file are the shape of the synthetic circuit
    full = S["full_counts"]
    assert (full["h"], full["l"], full["a"], full["b_g1"], full["b_g2"]) == (32767, 19955, 15598, 12402, 12402)
    sh = sy.CONF_SHAPE
    assert full["h"] == (1 << 15) - 1 and full["l"] == sh["n_aux"] and full["a"] == sh["n_inputs"] + sh["a_aux_density"] and full["b_g1"] == sh["b_density"]
