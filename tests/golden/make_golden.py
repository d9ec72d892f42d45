#!/usr/bin/env python3
"""Generates tests/golden/kats.json from the reference's own Rust test sources.

    python tests/golden/make_golden.py <checkout of LayerXcom/zero-chain>

The tests only read what this script writes under tests/golden/; they never need the reference itself.
Only numeric literals (known-answer vectors) are extracted — no reference code is copied.
For each listed `#[test] fn`, the ordered list of `FqRepr([..])` / `FrRepr([..])` limb groups
(little-endian u64 limbs as written in the source) is recorded; tests/test_oracle_kats.py
gives each list its meaning and cites the reference line range.

Also records SHA-256 digests and sizes of the reference's binary fixtures (the four 1000-point
encoding vector files and the shipped CRS files) so the oracle-generated equivalents can be
compared without committing the reference's files.
"""
import hashlib, json, os, re, sys

TESTS = {
    "fq.rs": ["test_fq_add_assign", "test_fq_sub_assign", "test_fq_mul_assign", "test_fq_squaring",
              "test_fq_double", "test_fq_negate", "test_fq_from_into_repr", "test_neg_one"],
    "fr.rs": ["test_fr_add_assign", "test_fr_sub_assign", "test_fr_mul_assign", "test_fr_squaring",
              "test_fr_double", "test_fr_negate", "test_fr_from_into_repr", "test_fr_root_of_unity"],
    "fq2.rs": ["test_fq2_squaring", "test_fq2_mul", "test_fq2_inverse", "test_fq2_addition",
               "test_fq2_subtraction", "test_fq2_negation", "test_fq2_doubling"],
    "ec.rs": ["test_g1_addition_correctness", "test_g1_doubling_correctness", "test_g1_same_y",
              "test_g2_addition_correctness", "test_g2_doubling_correctness"],
}
CONSTS = {   # named constants: (file, name) -> limb groups in the const's initializer
    "fq.rs": ["MODULUS", "R", "R2", "NEGATIVE_ONE", "B_COEFF", "G1_GENERATOR_X", "G1_GENERATOR_Y",
              "G2_GENERATOR_X_C0", "G2_GENERATOR_X_C1", "G2_GENERATOR_Y_C0", "G2_GENERATOR_Y_C1"],
    "fr.rs": ["MODULUS", "R", "R2", "GENERATOR", "ROOT_OF_UNITY"],
}
FILES = [
    "core/pairing/src/bls12_381/tests/g1_uncompressed_valid_test_vectors.dat",
    "core/pairing/src/bls12_381/tests/g1_compressed_valid_test_vectors.dat",
    "core/pairing/src/bls12_381/tests/g2_uncompressed_valid_test_vectors.dat",
    "core/pairing/src/bls12_381/tests/g2_compressed_valid_test_vectors.dat",
    "zface/params/conf_pk.dat", "zface/params/conf_vk.dat",
    "zface/params/anony_pk.dat",
    "core/bellman-verifier/src/tests/proving.params",
]
# points kept from each query of the shipped conf_pk.dat: about 1/32 of it, so the fixture stays small (the whole file is
# 10 MB).  The counts form a consistent proving key of a smaller circuit: h = 2^10 - 1, l = n_aux, a = 23 inputs + 486 aux.
SAMPLE_COUNTS = {"h": 1023, "l": 623, "a": 509, "b_g1": 387, "b_g2": 387}
GROUP = re.compile(r"F[qr]Repr\(\[\s*((?:0x[0-9a-fA-F_]+\s*,?\s*)+)\]\)")


def fn_body(src: str, name: str):
    m = re.search(r"fn\s+%s\s*\(\)\s*\{" % re.escape(name), src)
    assert m, name
    i = m.end(); depth = 1
    while depth:
        c = src[i]
        depth += (c == "{") - (c == "}")
        i += 1
    line = src.count("\n", 0, m.start()) + 1
    return src[m.end():i], line, src.count("\n", 0, i) + 1


def groups(text):
    out = []
    for g in GROUP.finditer(text):
        out.append([int(x.replace("_", ""), 16) for x in re.findall(r"0x[0-9a-fA-F_]+", g.group(1))])
    return out


def params_sample(pk):
    """The vk of `pk` unchanged (alpha .. delta, all ic points), then the first SAMPLE_COUNTS[q] points of every query q, in
    Parameters::write's grammar."""
    vk_len = 868 + 96 * int.from_bytes(pk[864:868], "big")
    out, off, full = bytearray(pk[:vk_len]), vk_len, {}
    for q, sz in (("h", 96), ("l", 96), ("a", 96), ("b_g1", 96), ("b_g2", 192)):
        n = int.from_bytes(pk[off:off + 4], "big")
        full[q] = n
        out += SAMPLE_COUNTS[q].to_bytes(4, "big") + pk[off + 4:off + 4 + sz * SAMPLE_COUNTS[q]]
        off += 4 + sz * n
    assert off == len(pk)
    return bytes(out), full


def main():
    REF = sys.argv[1]
    BLS = os.path.join(REF, "core/pairing/src/bls12_381")
    res = {"source": "LayerXcom/zero-chain core/pairing/src/bls12_381", "tests": {}, "consts": {}, "files": {}}
    for f, names in TESTS.items():
        src = open(os.path.join(BLS, f)).read()
        for n in names:
            body, l0, l1 = fn_body(src, n)
            res["tests"]["%s::%s" % (f, n)] = {"lines": [l0, l1], "groups": [[hex(v) for v in g] for g in groups(body)]}
    for f, names in CONSTS.items():
        src = open(os.path.join(BLS, f)).read()
        for n in names:
            m = re.search(r"const\s+%s\s*:[^=]*=\s*(.*?);" % n, src, re.S)
            assert m, (f, n)
            res["consts"]["%s::%s" % (f, n)] = [[hex(v) for v in g] for g in groups(m.group(1))]
    for p in FILES:
        b = open(os.path.join(REF, p), "rb").read()
        res["files"][p] = {"size": len(b), "sha256": hashlib.sha256(b).hexdigest()}
    # pairing known-answer: PreparedVerifyingKey.alpha_g1_beta_g2 = e(alpha_g1, beta_g2) as written by Fq12::write
    # (core/bellman-verifier/src/lib.rs:174-196) at conf_vk.dat[0:576]; alpha_g1 / beta_g2 from conf_pk.dat's vk header
    pk = open(os.path.join(REF, "zface/params/conf_pk.dat"), "rb").read()
    vk = open(os.path.join(REF, "zface/params/conf_vk.dat"), "rb").read()
    res["pairing_kat"] = {"alpha_g1_uncompressed": pk[0:96].hex(), "beta_g2_uncompressed": pk[192:384].hex(),
                          "alpha_g1_beta_g2_fq12": vk[0:576].hex(),
                          "source": "zface/params/conf_pk.dat[0:96], [192:384]; zface/params/conf_vk.dat[0:576]"}
    # a well-formed 192-byte proof held by the reference's own test (core/primitives/src/proof.rs:86-98): Proof::read must accept
    # it (flags, x < q, square roots, sign bits, subgroup membership of A, B, C) and Proof::write must give the same bytes back
    src = open(os.path.join(REF, "core/primitives/src/proof.rs")).read()
    m = re.search(r'fn test_proof_into_from\(\).*?hex!\("([0-9a-f]{384})"\)', src, re.S)
    assert m
    res["proof_kat"] = {"proof_hex": m.group(1), "source": "core/primitives/src/proof.rs:89 (test_proof_into_from)"}
    # verifier fixtures (binary, small): the shipped PreparedVerifyingKey files and the VerifyingKey head of the matching
    # proving keys (Parameters::write starts with vk: 868 bytes + 96 per ic point).  prepare_verifying_key of the latter
    # must reproduce the former byte for byte (tests/test_oracle_pairing.py, tests/test_gpu_verify.py).
    here = os.path.dirname(os.path.abspath(__file__))
    for name in ("conf", "anony"):
        pkb = open(os.path.join(REF, "zface/params/%s_pk.dat" % name), "rb").read()
        n_ic = int.from_bytes(pkb[864:868], "big")
        open(os.path.join(here, "%s_vk_head.bin" % name), "wb").write(pkb[:868 + 96 * n_ic])
        open(os.path.join(here, "%s_pvk.dat" % name), "wb").write(open(os.path.join(REF, "zface/params/%s_vk.dat" % name), "rb").read())
    # a sample of the shipped confidential-transfer CRS (10 133 592 B, 93 124 points): Parameters::read(&pk_buf[..], true)
    # (core/proofs/src/confidential.rs:95-103) is what the device loader replaces, and these points were not made by this
    # repository's code — tests/test_gpu_real_crs.py loads the sample, proves on it and round-trips it through zk_params_write
    sample, full = params_sample(open(os.path.join(REF, "zface/params/conf_pk.dat"), "rb").read())
    open(os.path.join(here, "conf_pk_sample.dat"), "wb").write(sample)
    res["conf_pk_sample"] = {"source": "zface/params/conf_pk.dat: its vk, then the first points of every query",
                             "full_counts": full, "counts": SAMPLE_COUNTS,
                             "size": len(sample), "sha256": hashlib.sha256(sample).hexdigest()}
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "kats.json")
    json.dump(res, open(out, "w"), indent=1)
    print("wrote", out, {k: len(v["groups"]) for k, v in res["tests"].items()})


if __name__ == "__main__":
    main()
