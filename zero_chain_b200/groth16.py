"""Host-side mirror of the reference's prover surface over the C ABI (include/zkb200.h).

Names follow upstream bellman 0.1.0 as the reference uses them:
  Parameters.read(buf, checked)      core/proofs/src/confidential.rs:99
  create_proof / create_random_proof core/proofs/src/confidential.rs:149, anonymous.rs:165
  multiexp(bases, exponents)         bellman::multiexp::multiexp  (SURVEY.md §3.2)
  EvaluationDomain.{fft,ifft,coset_fft,icoset_fft}   bellman::domain (SURVEY.md §8 a7)
  Proof (192-byte wire form)         core/bellman-verifier/src/lib.rs:40-110
  generate_random_parameters         core/proofs/src/setup.rs:28,59
Errors mirror bellman::SynthesisError (zface/src/error.rs:17,45-48).

All numeric arrays are numpy uint64 little-endian limbs: Fr canonical (n,4) at this boundary,
points in "limb form" (Montgomery x|y).  Everything computes on the GPU through libzkb200.so;
importing works without a GPU, any compute call without one raises ZkError(ZK_ERR_CUDA).
"""
from __future__ import annotations

import ctypes as C
import secrets

import numpy as np

from . import _lib
from ._lib import ZkError, check

R_MODULUS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


class SynthesisError(Exception):
    """bellman::SynthesisError variants reachable from the prover path."""
    NAMES = {-3: "AssignmentMissing", -4: "PolynomialDegreeTooLarge", -5: "UnexpectedIdentity", -6: "IoError",
             -7: "IoError(GroupDecodingError)", -8: "IoError(NotInField)", -9: "MalformedVerifyingKey", -10: "UnconstrainedVariable"}

    def __init__(self, code, msg):
        super().__init__("%s: %s" % (self.NAMES.get(code, "Error(%d)" % code), msg))
        self.code = code


def _ck(code):
    if code == 0:
        return
    msg = _lib.lib().zk_last_error().decode()
    if code in SynthesisError.NAMES:
        raise SynthesisError(code, msg)
    raise ZkError(code, msg)


def _u64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.reshape(shape) if shape is not None else a


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA device + stream (the analogue of bellman's multicore::Worker)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._h = C.c_void_p()
        _ck(_lib.lib().zk_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self._h)))
        self.device = device

    @property
    def stream(self) -> int:
        return _lib.lib().zk_ctx_stream(self._h) or 0

    def sync(self):
        _ck(_lib.lib().zk_ctx_sync(self._h))

    OPT_AFFINE_MIN_ENTRIES, OPT_AFFINE_LEVELS, OPT_VERIFY_LANES = 1, 2, 3

    def set_opt(self, opt: int, value: int):
        """zk_ctx_set_opt: tuning only (batched-affine threshold / rounds); results never depend on it."""
        _ck(_lib.lib().zk_ctx_set_opt(self._h, opt, value))

    def profile(self, enable: bool):
        _ck(_lib.lib().zk_ctx_profile(self._h, int(enable)))

    def profile_read(self):
        """(total ms, launches) of the dominant kernel since profile(True), CUDA events on this stream."""
        ms, n = C.c_double(), C.c_uint64()
        _ck(_lib.lib().zk_ctx_profile_read(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def profile_counts(self):
        """(G1 bucket additions, G2 bucket additions, G1 left to the XYZZ pass, G2 left to the XYZZ pass) executed by this
        context's MSMs (lanes included) since profile()."""
        v = [C.c_uint64() for _ in range(4)]
        _ck(_lib.lib().zk_ctx_profile_counts(self._h, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)

    def close(self):
        if self._h:
            _lib.lib().zk_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Bases:
    """Device-resident base points (+ window tables) for multiexp; group 1 = G1, 2 = G2."""

    def __init__(self, ctx: Context, group: int, limbs, window_bits: int = 0, precompute: bool = True):
        w = 12 if group == 1 else 24
        limbs = _u64(limbs, (-1, w))
        self.ctx, self.group, self.n = ctx, group, limbs.shape[0]
        self._h = C.c_void_p()
        _ck(_lib.lib().zk_bases_upload(ctx._h, group, _p(limbs), self.n, window_bits, int(precompute), C.byref(self._h)))
        self.window_bits = _lib.lib().zk_bases_window_bits(self._h)

    def free(self):
        if self._h:
            _lib.lib().zk_bases_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def multiexp(bases: Bases, exponents) -> bytes:
    """sum_i exponents[i] * bases[i]; exponents canonical (n,4) uint64 in HOST memory.
    Returns the uncompressed encoding (96 B G1 / 192 B G2)."""
    e = _u64(exponents, (-1, 4))
    out = np.zeros(96 if bases.group == 1 else 192, np.uint8)
    _ck(_lib.lib().zk_msm(bases.ctx._h, bases._h, _p(e), e.shape[0], _p(out)))
    return out.tobytes()


def multiexp_begin(ctx: Context, bases: Bases, exponents):
    """multiexp as a future (bellman's multiexp returns one): enqueue on `ctx`, collect with multiexp_end(ctx, bases).  `bases`
    may have been created through another context of the same device; alternate two contexts to pipeline successive MSMs."""
    e = _u64(exponents, (-1, 4))
    _ck(_lib.lib().zk_msm_begin(ctx._h, bases._h, _p(e), e.shape[0]))
    ctx._keep = e                         # the upload is asynchronous: keep the buffer alive until multiexp_end


def multiexp_device_begin(ctx: Context, bases: Bases, d_scalars_ptr: int, n: int):
    _ck(_lib.lib().zk_msm_device_begin(ctx._h, bases._h, C.c_void_p(d_scalars_ptr), n))


def multiexp_partial_device_begin(ctx: Context, bases: Bases, d_scalars_ptr: int, n: int, d_out_ptr: int):
    _ck(_lib.lib().zk_msm_partial_device_begin(ctx._h, bases._h, C.c_void_p(d_scalars_ptr), n, C.c_void_p(d_out_ptr)))


def points_fold_begin(ctx: Context, group: int, d_partials_ptr: int, count: int):
    _ck(_lib.lib().zk_points_fold_begin(ctx._h, group, C.c_void_p(d_partials_ptr), count))


def tail_stream(ctx: Context) -> int:
    """CUDA stream (high priority) on which a context finishes its futures; enqueue the all-gather of partials here."""
    return int(_lib.lib().zk_ctx_tail_stream(ctx._h))


def multiexp_end(ctx: Context, bases: Bases) -> bytes:
    out = np.zeros(96 if bases.group == 1 else 192, np.uint8)
    _ck(_lib.lib().zk_msm_end(ctx._h, _p(out)))
    ctx._keep = None
    return out.tobytes()


def multiexp_partial_device(bases: Bases, d_scalars_ptr: int, n: int, d_out_ptr: int):
    """Partial MSM result (XYZZ point, zk_partial_size bytes) left in device memory for the NCCL all-gather."""
    _ck(_lib.lib().zk_msm_partial_device(bases.ctx._h, bases._h, C.c_void_p(d_scalars_ptr), n, C.c_void_p(d_out_ptr)))


def points_fold(ctx: Context, group: int, d_partials_ptr: int, count: int) -> bytes:
    out = np.zeros(96 if group == 1 else 192, np.uint8)
    _ck(_lib.lib().zk_points_fold(ctx._h, group, C.c_void_p(d_partials_ptr), count, _p(out)))
    return out.tobytes()


def partial_size(group: int) -> int:
    return _lib.lib().zk_partial_size(group)


def multiexp_device(bases: Bases, d_scalars_ptr: int, n: int, batch: int = 1) -> bytes:
    out = np.zeros((96 if bases.group == 1 else 192) * batch, np.uint8)
    _ck(_lib.lib().zk_msm_batch_device(bases.ctx._h, bases._h, C.c_void_p(d_scalars_ptr), n, batch, _p(out)))
    return out.tobytes()


class EvaluationDomain:
    """Radix-2 domain over Fr; data are MONTGOMERY-form (n,4) uint64 arrays, natural order."""
    FFT, IFFT, COSET_FFT, ICOSET_FFT = 0, 1, 2, 3

    def __init__(self, ctx: Context, coeffs_mont):
        a = _u64(coeffs_mont, (-1, 4))
        m, exp = 1, 0
        while m < a.shape[0]:
            m *= 2
            exp += 1
            if exp >= 32:
                raise SynthesisError(-4, "PolynomialDegreeTooLarge")
        self.ctx, self.exp = ctx, exp
        self.coeffs = np.zeros((m, 4), np.uint64)
        self.coeffs[: a.shape[0]] = a

    def _run(self, mode):
        _ck(_lib.lib().zk_ntt_fr(self.ctx._h, _p(self.coeffs), self.exp, mode))
        return self

    def fft(self): return self._run(self.FFT)
    def ifft(self): return self._run(self.IFFT)
    def coset_fft(self): return self._run(self.COSET_FFT)
    def icoset_fft(self): return self._run(self.ICOSET_FFT)


class Parameters:
    """groth16::Parameters<Bls12> held on the device."""

    def __init__(self, ctx: Context, handle, counts):
        self.ctx, self._h = ctx, handle
        self.n_ic, self.n_h, self.n_l, self.n_a, self.n_b_g1, self.n_b_g2 = counts

    @staticmethod
    def read(ctx: Context, buf: bytes, checked: bool = True) -> "Parameters":
        b = np.frombuffer(buf, np.uint8)
        h = C.c_void_p()
        _ck(_lib.lib().zk_params_load(ctx._h, _p(b), len(buf), int(checked), C.byref(h)))
        cnt = np.zeros(6, np.uint64)
        _ck(_lib.lib().zk_params_counts(h, _p(cnt)))
        return Parameters(ctx, h, [int(x) for x in cnt])

    @staticmethod
    def read_cached(ctx: Context, buf: bytes, cache_path: str) -> "Parameters":
        """Parameters::read(buf, true) through the decoded-CRS cache on disk (zk_params_load_cached); `.cache_hit` tells which
        path ran.  The reference re-reads and re-checks the whole proving key on every start (crypto_components.rs:320-328)."""
        b = np.frombuffer(buf, np.uint8)
        h, hit = C.c_void_p(), C.c_int(0)
        _ck(_lib.lib().zk_params_load_cached(ctx._h, _p(b), len(buf), cache_path.encode(), C.byref(hit), C.byref(h)))
        cnt = np.zeros(6, np.uint64)
        _ck(_lib.lib().zk_params_counts(h, _p(cnt)))
        prm = Parameters(ctx, h, [int(x) for x in cnt])
        prm.cache_hit = bool(hit.value)
        return prm

    def write(self) -> bytes:
        """Parameters::write (core/proofs/src/confidential.rs:83): the resident CRS as the exact byte stream `read` consumes."""
        out = np.zeros(int(_lib.lib().zk_params_size(self._h)), np.uint8)
        _ck(_lib.lib().zk_params_write(self.ctx._h, self._h, _p(out)))
        return out.tobytes()

    def vk_bytes(self) -> bytes:
        """VerifyingKey::write of `params.vk` (core/proofs/src/setup.rs:31): the head of the Parameters stream."""
        out = np.zeros(int(_lib.lib().zk_params_vk_size(self._h)), np.uint8)
        _ck(_lib.lib().zk_params_write_vk(self.ctx._h, self._h, _p(out)))
        return out.tobytes()

    def free(self):
        if self._h:
            _lib.lib().zk_params_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PreparedVerifyingKey:
    """bellman_verifier::PreparedVerifyingKey<Bls12> on the device (core/bellman-verifier/src/lib.rs:110-245)."""

    def __init__(self, ctx: Context, handle):
        self.ctx, self._h = ctx, handle
        self.num_inputs = int(_lib.lib().zk_pvk_num_inputs(handle))

    @staticmethod
    def read(ctx: Context, buf: bytes) -> "PreparedVerifyingKey":
        """PreparedVerifyingKey::read — the bytes of zface/params/conf_vk.dat."""
        b = np.frombuffer(buf, np.uint8)
        h = C.c_void_p()
        _ck(_lib.lib().zk_pvk_load(ctx._h, _p(b), len(buf), C.byref(h)))
        return PreparedVerifyingKey(ctx, h)

    @staticmethod
    def prepare(ctx: Context, vk_bytes: bytes) -> "PreparedVerifyingKey":
        """prepare_verifying_key(&vk) (verifier.rs:15-30); vk_bytes = VerifyingKey encoding / head of Parameters::write."""
        b = np.frombuffer(vk_bytes, np.uint8)
        h = C.c_void_p()
        _ck(_lib.lib().zk_pvk_prepare(ctx._h, _p(b), len(vk_bytes), C.byref(h)))
        return PreparedVerifyingKey(ctx, h)

    def write(self) -> bytes:
        out = np.zeros(int(_lib.lib().zk_pvk_size(self._h)), np.uint8)
        _ck(_lib.lib().zk_pvk_write(self._h, _p(out)))
        return out.tobytes()

    def free(self):
        if self._h:
            _lib.lib().zk_pvk_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


VERDICT_OK, VERDICT_FALSE, VERDICT_INVALID_DATA, VERDICT_POINT_INFINITY = 1, 0, 2, 3


def verify_proofs(pvk: PreparedVerifyingKey, proofs: bytes, public_inputs) -> list:
    """Proof::read + verify_proof (verifier.rs:32-63) for len(proofs)/192 proofs; public_inputs: one list of ints per
    proof (without the leading ONE).  Returns the verdict codes of include/zkb200.h; raises
    SynthesisError(MalformedVerifyingKey) when the input count does not match the key."""
    n = len(proofs) // 192
    assert len(proofs) == 192 * n and len(public_inputs) == n
    n_in = len(public_inputs[0]) if n else pvk.num_inputs
    assert all(len(x) == n_in for x in public_inputs)
    inp = _u64([_fr_limbs(v) for row in public_inputs for v in row]) if n * n_in else np.zeros(1, np.uint64)
    pb = np.frombuffer(proofs, np.uint8) if n else np.zeros(1, np.uint8)
    out = np.zeros(max(n, 1), np.uint8)
    _ck(_lib.lib().zk_groth16_verify_batch(pvk.ctx._h, pvk._h, n, _p(pb), _p(inp), n_in, _p(out)))
    return [int(v) for v in out[:n]]


def verify_proof(pvk: PreparedVerifyingKey, proof: bytes, public_inputs) -> bool:
    """verify_proof(pvk, proof, inputs) -> Ok(bool); a proof that Proof::read rejects raises ZkError (io::Error there)."""
    v = verify_proofs(pvk, proof, [list(public_inputs)])[0]
    if v >= 2:
        raise ZkError(-7, "Proof::read: %s" % ("PointInfinity" if v == 3 else "InvalidData"))
    return v == 1


def verify_proofs_device(pvk: PreparedVerifyingKey, n: int, d_proofs_ptr: int, d_inputs_ptr: int, n_inputs: int, d_verdicts_ptr: int):
    _ck(_lib.lib().zk_groth16_verify_batch_device(pvk.ctx._h, pvk._h, n, C.c_void_p(d_proofs_ptr), C.c_void_p(d_inputs_ptr), n_inputs,
                                                  C.c_void_p(d_verdicts_ptr)))


def pairing(ctx: Context, g1_uncompressed: bytes, g2_uncompressed: bytes) -> bytes:
    """Engine::pairing for len/96 pairs; 576 bytes each in Fq12::write order."""
    n = len(g1_uncompressed) // 96
    assert len(g1_uncompressed) == 96 * n and len(g2_uncompressed) == 192 * n
    out = np.zeros(576 * max(n, 1), np.uint8)
    _ck(_lib.lib().zk_pairing_batch(ctx._h, n, _p(np.frombuffer(g1_uncompressed, np.uint8)), _p(np.frombuffer(g2_uncompressed, np.uint8)), _p(out)))
    return out[:576 * n].tobytes()


class Proof:
    """zerochain_primitives::Proof(Vec<u8>) — the wire wrapper of the 192 proof bytes (core/primitives/src/proof.rs:12-62): the
    runtime moves `Proof` SCALE-encoded (parity_codec derive: Compact<u32> length, then the bytes) and converts to / from
    bellman_verifier::Proof with Proof::read / Proof::write.  Pure byte handling: nothing here touches the device."""
    SIZE = 192

    def __init__(self, raw: bytes):
        self._b = bytes(raw)

    @staticmethod
    def from_slice(raw: bytes) -> "Proof":
        return Proof(raw)

    def as_bytes(self) -> bytes:
        return self._b

    def encode(self) -> bytes:
        """parity_codec::Encode of Vec<u8>: compact length prefix (single / two / four-byte mode), then the bytes."""
        n = len(self._b)
        if n < 1 << 6:
            pre = bytes([n << 2])
        elif n < 1 << 14:
            pre = ((n << 2) | 1).to_bytes(2, "little")
        else:
            assert n < 1 << 30
            pre = ((n << 2) | 2).to_bytes(4, "little")
        return pre + self._b

    @staticmethod
    def decode(buf: bytes) -> "Proof":
        mode = buf[0] & 3
        if mode == 0:
            n, off = buf[0] >> 2, 1
        elif mode == 1:
            n, off = int.from_bytes(buf[:2], "little") >> 2, 2
        elif mode == 2:
            n, off = int.from_bytes(buf[:4], "little") >> 2, 4
        else:
            raise ValueError("big-integer compact lengths do not occur for proofs")
        if len(buf) < off + n:
            raise ValueError("truncated Proof")
        return Proof(buf[off:off + n])

    def __eq__(self, other):
        return isinstance(other, Proof) and self._b == other._b

    def __str__(self):
        return "0x" + self._b.hex()


class ProvingAssignment:
    """What bellman's ProvingAssignment holds after `circuit.synthesize` and the input rows
    (SURVEY.md §3.2): per-constraint evaluations, assignments and the three density maps."""

    def __init__(self, a, b, c, input_assignment, aux_assignment, a_aux_density, b_input_density, b_aux_density):
        self.a, self.b, self.c = (_u64(x, (-1, 4)) for x in (a, b, c))
        self.input_assignment = _u64(input_assignment, (-1, 4))
        self.aux_assignment = _u64(aux_assignment, (-1, 4))
        self.a_aux_density = np.ascontiguousarray(a_aux_density, np.uint8)
        self.b_input_density = np.ascontiguousarray(b_input_density, np.uint8)
        self.b_aux_density = np.ascontiguousarray(b_aux_density, np.uint8)


def _fr_limbs(x: int):
    return np.array([(x >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)], np.uint64)


def create_proof(prover: ProvingAssignment, params: Parameters, r: int, s: int) -> bytes:
    """groth16::create_proof(circuit, params, r, s) below synthesis -> Proof::write bytes (192 B)."""
    out = np.zeros(192, np.uint8)
    rr, ss = _fr_limbs(r), _fr_limbs(s)
    L = _lib.lib()
    _ck(L.zk_groth16_prove(params.ctx._h, params._h, _p(prover.a), _p(prover.b), _p(prover.c), prover.a.shape[0],
                           _p(prover.input_assignment), prover.input_assignment.shape[0],
                           _p(prover.aux_assignment), prover.aux_assignment.shape[0],
                           _p(prover.a_aux_density), _p(prover.b_input_density), _p(prover.b_aux_density),
                           _p(rr), _p(ss), _p(out)))
    return out.tobytes()


def create_random_proof(prover: ProvingAssignment, params: Parameters, rng=None) -> bytes:
    """groth16::create_random_proof: draws r, s uniformly in Fr (Fr::rand, fr.rs:255-267) then create_proof."""
    draw = (lambda: secrets.randbelow(R_MODULUS)) if rng is None else (lambda: rng.randrange(R_MODULUS))
    return create_proof(prover, params, draw(), draw())


def create_proof_batch(provers, params: Parameters, rs, ss) -> bytes:
    """`len(provers)` witnesses of the same circuit in one device pass; returns batch*192 bytes."""
    p0 = provers[0]
    batch = len(provers)
    cat = lambda name: np.ascontiguousarray(np.concatenate([getattr(p, name) for p in provers], axis=0))
    a, b, c, inp, aux = (cat(k) for k in ("a", "b", "c", "input_assignment", "aux_assignment"))
    rr = np.stack([_fr_limbs(x) for x in rs]); sv = np.stack([_fr_limbs(x) for x in ss])
    out = np.zeros(192 * batch, np.uint8)
    _ck(_lib.lib().zk_groth16_prove_batch(params.ctx._h, params._h, batch, _p(a), _p(b), _p(c), p0.a.shape[0],
                                          _p(inp), p0.input_assignment.shape[0], _p(aux), p0.aux_assignment.shape[0],
                                          _p(p0.a_aux_density), _p(p0.b_input_density), _p(p0.b_aux_density),
                                          _p(rr), _p(sv), _p(out)))
    return out.tobytes()


class ConstraintSystem:
    """The fixed R1CS of a circuit resident on the device (CSR), so proofs can be made straight from assignments
    (zk_groth16_prove_witness_batch).  rows_*: per constraint a list of (variable, coefficient) with variable < n_inputs
    for inputs and n_inputs + i for aux i — the at/bt/ct that bellman's KeypairAssembly collects."""

    def __init__(self, ctx: Context, n_inputs: int, n_aux: int, rows_a, rows_b, rows_c):
        self.ctx, self.n_inputs, self.n_aux = ctx, n_inputs, n_aux
        n_c = len(rows_a)
        assert len(rows_b) == n_c and len(rows_c) == n_c
        arrs = []
        for rows in (rows_a, rows_b, rows_c):
            rp = np.zeros(n_c + 1, np.uint32)
            rp[1:] = np.cumsum([len(r) for r in rows])
            col = np.array([v for r in rows for v, _ in r] or [0], np.uint32)
            cf = np.zeros((max(1, int(rp[-1])), 4), np.uint64)
            k = 0
            for r in rows:
                for _, c in r:
                    for j in range(4):
                        cf[k, j] = (c >> (64 * j)) & 0xFFFFFFFFFFFFFFFF
                    k += 1
            arrs += [rp, col, cf]
        self._h = C.c_void_p()
        _ck(_lib.lib().zk_r1cs_load(ctx._h, n_c, n_inputs, n_aux, *[_p(a) for a in arrs], C.byref(self._h)))

    def free(self):
        if self._h:
            _lib.lib().zk_r1cs_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def create_proof_from_witness_batch(cs: ConstraintSystem, params: Parameters, batch: int, inputs, aux, r, s) -> bytes:
    """inputs [batch][n_inputs][4], aux [batch][n_aux][4] canonical; r, s [batch][4] -> batch * 192 bytes."""
    inputs, aux = _u64(inputs, (batch, cs.n_inputs, 4)), _u64(aux, (batch, cs.n_aux, 4))
    r, s = _u64(r, (batch, 4)), _u64(s, (batch, 4))
    out = np.zeros(192 * batch, np.uint8)
    _ck(_lib.lib().zk_groth16_prove_witness_batch(params.ctx._h, params._h, cs._h, batch, _p(inputs), _p(aux), _p(r), _p(s), _p(out)))
    return out.tobytes()


def generate_parameters(cs: ConstraintSystem, g1: bytes, g2: bytes, alpha: int, beta: int, gamma: int, delta: int, tau: int) -> Parameters:
    """groth16::generate_parameters(circuit, g1, g2, alpha, beta, gamma, delta, tau) for the constraint system `cs` on its device.
    g1 / g2: G1Uncompressed (96 B) / G2Uncompressed (192 B) generators; the five scalars canonical.  The result is resident and ready
    to prove with; its write() is the byte stream bellman's Parameters::write emits for the same inputs."""
    g1, g2 = np.frombuffer(bytes(g1), np.uint8), np.frombuffer(bytes(g2), np.uint8)
    assert g1.size == 96 and g2.size == 192
    sc = [_fr_limbs(x) if 0 <= x < 1 << 256 else None for x in (alpha, beta, gamma, delta, tau)]
    if any(x is None for x in sc):
        raise SynthesisError(-8, "scalar outside [0, 2^256)")
    h = C.c_void_p()
    _ck(_lib.lib().zk_groth16_generate(cs.ctx._h, cs._h, _p(g1), _p(g2), *[_p(x) for x in sc], C.byref(h)))
    cnt = np.zeros(6, np.uint64)
    _ck(_lib.lib().zk_params_counts(h, _p(cnt)))
    return Parameters(cs.ctx, h, [int(x) for x in cnt])


def generate_random_parameters(cs: ConstraintSystem, rng=None) -> Parameters:
    """groth16::generate_random_parameters: g1, g2 uniform non-identity group elements (random non-zero multiples of the
    standard generators, which is what G1::rand / G2::rand give in a group of prime order), then alpha, beta, gamma, delta, tau
    uniform in Fr (Fr::rand), drawn in bellman's order; `rng` as for create_random_proof."""
    from .synthetic import g1_limbs_to_uncompressed, g2_limbs_to_uncompressed
    draw = (lambda: secrets.randbelow(R_MODULUS)) if rng is None else (lambda: rng.randrange(R_MODULUS))
    k1, k2 = 1 + draw() % (R_MODULUS - 1), 1 + draw() % (R_MODULUS - 1)
    g1 = g1_limbs_to_uncompressed(scalar_mul_many(cs.ctx, 1, G1_GENERATOR, [_fr_limbs(k1)])[0])
    g2 = g2_limbs_to_uncompressed(scalar_mul_many(cs.ctx, 2, G2_GENERATOR, [_fr_limbs(k2)])[0])
    alpha, beta, gamma, delta, tau = (draw() for _ in range(5))
    return generate_parameters(cs, g1, g2, alpha, beta, gamma, delta, tau)


def parameter_files(params: Parameters):
    """The two files of the reference's write_to_file (core/proofs/src/crypto_components.rs:277): the proving key
    (Parameters::write, e.g. conf_pk.dat) and the prepared verifying key (PreparedVerifyingKey::write of
    prepare_verifying_key(&params.vk), e.g. conf_vk.dat)."""
    pvk = PreparedVerifyingKey.prepare(params.ctx, params.vk_bytes())
    try:
        return params.write(), pvk.write()
    finally:
        pvk.free()


def create_proof_batch_raw(params: Parameters, batch: int, a, b, c, inputs, aux, a_aux_density, b_input_density, b_aux_density, r, s) -> bytes:
    """Same as create_proof_batch with the per-proof arrays already concatenated ([batch][n][4] uint64, e.g. views
    of pinned host memory): exactly one zk_groth16_prove_batch call, no host-side copies."""
    a, b, c, inputs, aux = (_u64(x, (batch, -1, 4)) for x in (a, b, c, inputs, aux))
    r, s = _u64(r, (batch, 4)), _u64(s, (batch, 4))
    d1, d2, d3 = (np.ascontiguousarray(x, np.uint8) for x in (a_aux_density, b_input_density, b_aux_density))
    out = np.zeros(192 * batch, np.uint8)
    _ck(_lib.lib().zk_groth16_prove_batch(params.ctx._h, params._h, batch, _p(a), _p(b), _p(c), a.shape[1],
                                          _p(inputs), inputs.shape[1], _p(aux), aux.shape[1], _p(d1), _p(d2), _p(d3), _p(r), _p(s), _p(out)))
    return out.tobytes()


# ---- utilities ---------------------------------------------------------------------------------------
def scalar_mul_many(ctx: Context, group: int, base_limbs, scalars):
    s = _u64(scalars, (-1, 4))
    w = 12 if group == 1 else 24
    base = _u64(base_limbs, (w,))
    out = np.zeros((s.shape[0], w), np.uint64)
    _ck(_lib.lib().zk_scalar_mul_many(ctx._h, group, _p(base), _p(s), s.shape[0], _p(out)))
    return out


FIELD_FQ, FIELD_FR = 0, 1
OP_MUL, OP_ADD, OP_SUB, OP_SQR, OP_INV, OP_FROM_REPR, OP_INTO_REPR = range(7)


def field_op(ctx: Context, field: int, op: int, a, b=None):
    nl = 6 if field == 0 else 4
    a = _u64(a, (-1, nl))
    bb = None if b is None else _u64(b, (-1, nl))
    out = np.zeros_like(a)
    _ck(_lib.lib().zk_field_op(ctx._h, field, op, _p(a), _p(bb) if bb is not None else None, a.shape[0], _p(out)))
    return out


def bench_modmul(ctx: Context, field: int, blocks: int, threads: int, iters: int):
    per_s, ms = C.c_double(), C.c_double()
    _ck(_lib.lib().zk_bench_modmul(ctx._h, field, blocks, threads, iters, C.byref(per_s), C.byref(ms)))
    return per_s.value, ms.value


# constants of the generators in limb form (Montgomery; fq.rs:85-136) for building synthetic inputs
G1_GENERATOR = np.array([0x5cb38790fd530c16, 0x7817fc679976fff5, 0x154f95c7143ba1c1, 0xf0ae6acdf3d0e747, 0xedce6ecc21dbf440, 0x120177419e0bfb75,
                         0xbaac93d50ce72271, 0x8c22631a7918fd8e, 0xdd595f13570725ce, 0x51ac582950405194, 0x0e1c8c3fad0059c0, 0x0bbc3efc5008a26a], np.uint64)
G2_GENERATOR = np.array([0xf5f28fa202940a10, 0xb3f5fb2687b4961a, 0xa1a893b53e2ae580, 0x9894999d1a3caee9, 0x6f67b7631863366b, 0x058191924350bcd7,
                         0xa5a9c0759e23f606, 0xaaa0c59dbccd60c3, 0x3bb17e18e2867806, 0x1b1ab6cc8541b367, 0xc2b6ed0ef2158547, 0x11922a097360edf3,
                         0x4c730af860494c4a, 0x597cfa1f5e369c5a, 0xe7e6856caa0a635a, 0xbbefb5e96e0d495f, 0x07d3a975f0ef25a2, 0x0083fd8e7e80dae5,
                         0xadc0fc92df64b05d, 0x18aa270a2b1461dc, 0x86adac6a3be4eba0, 0x79495c4ec93da33a, 0xe7175850a43ccaed, 0x0b2bc2a163de1bf2], np.uint64)
