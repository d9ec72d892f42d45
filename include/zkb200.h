/* zkb200 — C ABI of the B200-native Groth16 prover hot path (libzkb200.so).
 *
 * Drop-in boundary for the path LayerXcom/zero-chain reaches through
 *     bellman::groth16::create_random_proof(circuit, &Parameters<Bls12>, rng)
 * (call sites core/proofs/src/confidential.rs:149, core/proofs/src/anonymous.rs:165; the CRS is
 * read at core/proofs/src/confidential.rs:95-103 by Parameters::read(buf, checked = true)).
 * bellman 0.1.0 itself is an un-vendored dependency (Cargo.lock:210-212), so each entry point
 * cites the upstream function it replaces and the reference call site that reaches it.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every input/output buffer for the duration
 *     of the call; handles (zk_ctx, zk_bases, zk_params) are owned by the library.
 *   - Fr scalars cross the ABI as canonical FrRepr: 4 little-endian u64 limbs, value < r
 *     (= Fr::into_repr(), core/pairing/src/bls12_381/fr.rs:290-303).  Montgomery form is internal.
 *   - the CRS crosses once as the exact Parameters::write byte stream (zface/params/conf_pk.dat);
 *     proofs come back as the exact Proof::write bytes (core/bellman-verifier/src/lib.rs:55-65).
 *   - "limb form" points (kernel-level entry points only): affine x|y in Montgomery limbs,
 *     96 B (G1: x[6] y[6] u64) or 192 B (G2: x.c0 x.c1 y.c0 y.c1), infinity = all zero.
 *   - every function returns ZK_OK (0) or a negative error; zk_last_error() gives the text.
 *     Error codes mirror bellman's SynthesisError / io::Error as seen at the call sites
 *     (zface/src/error.rs:17,45-48).
 *   - thread safety: a zk_ctx is single-threaded (one CUDA stream + its own workspace, NTT tables and lanes); zk_params /
 *     zk_bases / zk_pvk / zk_r1cs are read-only after creation and may be shared by several contexts on the same device.
 *     Concurrent proving on one zk_params (what bellman's Arc<Vec<..>> parameters allow, SURVEY.md §8b) = one zk_ctx per
 *     host thread, all passing the same zk_params (bench.py's two_batches_in_flight does exactly that).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     ZK_ERR_CUDA.
 */
#ifndef ZKB200_H
#define ZKB200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ZK_OK 0
#define ZK_ERR_CUDA (-1)                 /* no device / CUDA runtime failure */
#define ZK_ERR_INVALID (-2)              /* bad argument */
#define ZK_ERR_ASSIGNMENT_MISSING (-3)   /* SynthesisError::AssignmentMissing: vector sizes do not match the CRS */
#define ZK_ERR_POLY_DEGREE_TOO_LARGE (-4)/* SynthesisError::PolynomialDegreeTooLarge */
#define ZK_ERR_UNEXPECTED_IDENTITY (-5)  /* SynthesisError::UnexpectedIdentity (base or delta at infinity) */
#define ZK_ERR_IO (-6)                   /* SynthesisError::IoError: truncated / malformed Parameters stream */
#define ZK_ERR_DECODE (-7)               /* GroupDecodingError (not on curve, not in subgroup, bad flags, x >= q) */
#define ZK_ERR_NOT_CANONICAL (-8)        /* a scalar >= r (PrimeFieldDecodingError::NotInField) */
#define ZK_ERR_MALFORMED_VK (-9)         /* SynthesisError::MalformedVerifyingKey: inputs.len() + 1 != ic.len() */
#define ZK_ERR_UNCONSTRAINED_VARIABLE (-10)  /* SynthesisError::UnconstrainedVariable: an L-query point is the identity */

const char *zk_last_error(void);
int zk_device_count(void);
const char *zk_version(void);

/* ---- execution context: one per (device, stream) ------------------------------------------- */
typedef struct zk_ctx zk_ctx;
/* stream: a cudaStream_t to run on (e.g. the caller's current stream) or NULL to create one. */
int zk_ctx_create(int device, void *stream, zk_ctx **out);
void zk_ctx_destroy(zk_ctx *ctx);
int zk_ctx_sync(zk_ctx *ctx);
/* Tuning options of a context (and of the prover lanes it owns).  Results never depend on them.
 *   ZK_OPT_AFFINE_MIN_ENTRIES  MSMs with at least this many (term, window) entries reduce their buckets with batched-affine
 *                              rounds (6.4 field products per addition instead of 10, one shared inversion per round, ~0.2 ms of
 *                              latency each) before the XYZZ pass: +8 % MSM throughput with two MSMs in flight, +13 % for a
 *                              256-proof batch, -3 % on one blocking 2^20 MSM (profiles/r02_experiments.md).  Default 2^22;
 *                              -1 = never, 0 = always.
 *   ZK_OPT_AFFINE_LEVELS       number of rounds; -1 (default) = from the average bucket length.
 *   ZK_OPT_VERIFY_LANES        1 (default): the verifier's Miller loops and final exponentiations spread every Fq12 value over six
 *                              lanes of a warp; 0: one thread per proof (the round-1 kernels, kept as the A/B reference). */
#define ZK_OPT_AFFINE_MIN_ENTRIES 1
#define ZK_OPT_AFFINE_LEVELS 2
#define ZK_OPT_VERIFY_LANES 3
int zk_ctx_set_opt(zk_ctx *ctx, int opt, long value);
void *zk_ctx_stream(zk_ctx *ctx);

/* ---- multi-scalar multiplication (replaces bellman::multiexp::multiexp, SURVEY.md §8 a8) ----- */
typedef struct zk_bases zk_bases;
/* Upload n affine bases (limb form, HOST memory) and, if precompute != 0, build the window tables
 * 2^(c*w) * P_i on the device (the CRS is fixed, so this is done once, like Parameters::read).
 * window_bits = 0 picks c from n.  group = 1 (G1) or 2 (G2).  Infinity bases are rejected
 * (bellman: SynthesisError::UnexpectedIdentity). */
int zk_bases_upload(zk_ctx *ctx, int group, const uint64_t *bases_limbs, size_t n, int window_bits, int precompute,
                    zk_bases **out);
void zk_bases_free(zk_bases *b);
size_t zk_bases_len(const zk_bases *b);
int zk_bases_window_bits(const zk_bases *b);
/* sum_i scalars[i] * P_i over the first n bases.  scalars: canonical FrRepr in HOST memory
 * (host -> device copy is part of the call); out: uncompressed encoding (96 B for G1, 192 B for G2;
 * G1Uncompressed / G2Uncompressed::from_affine, core/pairing/src/bls12_381/ec.rs:686-752, 1343-1425). */
int zk_msm(zk_ctx *ctx, const zk_bases *b, const uint64_t *scalars, size_t n, uint8_t *out);
/* same with scalars already resident in DEVICE memory (kernel-only timing; prover-internal use) */
int zk_msm_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, uint8_t *out);
/* The same MSM as a future, which is what bellman's multiexp returns (multiexp.rs: Box<Future<Item = G>>): begin enqueues the
 * upload (host variant), the MSM, the affine conversion and the download of the encoded point, and returns; end waits and
 * hands out the 96 / 192 bytes.  One MSM may be in flight per context.  Everything after the bucket accumulation runs on a
 * high-priority stream of the context, so two contexts used alternately overlap the latency-bound tail of one MSM (and the
 * upload of the next scalars) with the accumulation of the other — results are identical to zk_msm / zk_msm_device. */
int zk_msm_begin(zk_ctx *ctx, const zk_bases *b, const uint64_t *scalars, size_t n);
int zk_msm_device_begin(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n);
int zk_msm_end(zk_ctx *ctx, uint8_t *out);
/* multi-GPU form: the rank's partial (zk_partial_size bytes) lands in d_partial_out on zk_ctx_tail_stream(ctx); the caller enqueues
 * its all-gather on that stream, then zk_points_fold_begin (fold + encode + download on the same stream); zk_msm_end collects. */
void *zk_ctx_tail_stream(zk_ctx *ctx);
int zk_msm_partial_device_begin(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, void *d_partial_out);
int zk_points_fold_begin(zk_ctx *ctx, int group, const void *d_partials, size_t count);
/* batch of `batch` independent scalar vectors (each n long, contiguous) against the same bases;
 * out: batch encodings.  Used by the batched prover. */
int zk_msm_batch_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, size_t batch, uint8_t *out);
/* multi-GPU helper: the partial result as an XYZZ point in DEVICE memory is all-gathered by the
 * caller (NCCL, bytes) and folded with zk_points_fold: out = encoding of sum of `count` device
 * points of zk_partial_size(group) bytes each. */
size_t zk_partial_size(int group);
int zk_msm_partial_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, void *d_partial_out);
int zk_points_fold(zk_ctx *ctx, int group, const void *d_partials, size_t count, uint8_t *out);

/* ---- Fr radix-2 NTT (replaces bellman::domain::EvaluationDomain, SURVEY.md §8 a7) ----------- */
#define ZK_NTT_FFT 0         /* EvaluationDomain::fft        */
#define ZK_NTT_IFFT 1        /* EvaluationDomain::ifft       (includes the m^-1 scaling) */
#define ZK_NTT_COSET_FFT 2   /* EvaluationDomain::coset_fft  (distribute_powers(7) then fft) */
#define ZK_NTT_ICOSET_FFT 3  /* EvaluationDomain::icoset_fft (ifft then distribute_powers(7^-1)) */
/* data: 2^log_n Fr elements, MONTGOMERY limbs (the in-memory form of bellman's Scalar<E>), natural
 * order in and out, transformed in place.  Host-memory and device-memory flavours. */
int zk_ntt_fr(zk_ctx *ctx, uint64_t *data, unsigned log_n, int mode);
int zk_ntt_fr_device(zk_ctx *ctx, void *d_data, unsigned log_n, int mode);

/* ---- Groth16 (replaces bellman::groth16::{Parameters::read, create_proof}) ------------------ */
typedef struct zk_params zk_params;
/* Parses the exact Parameters::write stream (SURVEY.md §3.3; reference call
 * core/proofs/src/confidential.rs:99 `Parameters::read(&buf[..], true)`), decodes every point on
 * the device, with checked != 0 also tests on-curve and r-torsion membership
 * (core/pairing/src/bls12_381/ec.rs:675-685), rejects infinity in the query vectors, and keeps the
 * CRS (and its MSM window tables) resident on the context's device. */
int zk_params_load(zk_ctx *ctx, const uint8_t *pk_bytes, size_t len, int checked, zk_params **out);
void zk_params_free(zk_params *p);
/* counts[6] = { ic, h, l, a, b_g1, b_g2 } */
int zk_params_counts(const zk_params *p, uint64_t counts[6]);
/* Parameters::write (bellman groth16; reference call core/proofs/src/confidential.rs:73-93 `self.proving_key.write(..)`): the
 * resident CRS re-encoded as the exact byte stream Parameters::read consumes — zk_params_size bytes; loading a file and writing
 * it back reproduces the file byte for byte.  zk_params_write_vk emits only the VerifyingKey head (VerifyingKey::write: alpha_g1 |
 * beta_g1 | beta_g2 | gamma_g2 | delta_g1 | delta_g2 | u32 n | ic; zk_params_vk_size bytes) — what `params.vk`
 * (core/proofs/src/setup.rs:31, prepare_verifying_key(&params.vk)) needs on the host side. */
size_t zk_params_size(const zk_params *p);
size_t zk_params_vk_size(const zk_params *p);
int zk_params_write(zk_ctx *ctx, const zk_params *p, uint8_t *out);
int zk_params_write_vk(zk_ctx *ctx, const zk_params *p, uint8_t *out);
/* Parameters::read(buf, checked = true) with a decoded-CRS cache on disk (SURVEY.md §8 f1; the "FIX: too heavy" read at
 * core/proofs/src/crypto_components.rs:320-328).  If `cache_path` holds the decoded Montgomery points of exactly these bytes
 * (SHA-256 of the whole stream, length and vector counts are compared, and the cached points carry their own SHA-256), they are uploaded as they are — no decoding, no on-curve
 * or subgroup tests (*cache_hit = 1).  Otherwise the stream goes through the full CHECKED load and the cache file is (re)written
 * atomically (*cache_hit = 0); a cache that cannot be written is not an error.  cache_hit may be NULL.
 * Trust: the hashes guard against corruption and against a cache of another key, not against an adversary who can write
 * `cache_path` (they could store off-curve points with a matching body hash) — keep the file where the proving key itself lives. */
int zk_params_load_cached(zk_ctx *ctx, const uint8_t *pk_bytes, size_t len, const char *cache_path, int *cache_hit, zk_params **out);

/* create_proof for ONE already-synthesised witness (the Rust shim runs ProvingAssignment::synthesize
 * and the `input_i * 0 = 0` rows, then calls this; SURVEY.md §8b).
 *   a/b/c_evals      n_constraints canonical Fr each (<A_j,z>, <B_j,z>, <C_j,z>)
 *   input_assignment n_inputs canonical Fr, [0] = ONE;  aux_assignment n_aux canonical Fr
 *   *_density        one BYTE per variable (0/1): DensityTracker bits of the A-aux, B-input, B-aux queries
 *   r, s             the two blinding scalars create_random_proof draws (canonical)
 *   proof_out        192 B = Proof::write (compressed A | B | C) */
int zk_groth16_prove(zk_ctx *ctx, const zk_params *p,
                     const uint64_t *a_evals, const uint64_t *b_evals, const uint64_t *c_evals, size_t n_constraints,
                     const uint64_t *input_assignment, size_t n_inputs,
                     const uint64_t *aux_assignment, size_t n_aux,
                     const uint8_t *a_aux_density, const uint8_t *b_input_density, const uint8_t *b_aux_density,
                     const uint64_t r[4], const uint64_t s[4], uint8_t proof_out[192]);
/* `batch` witnesses of the same circuit (same sizes and densities), arrays concatenated per proof:
 * a_evals[batch][n_constraints][4] ... r[batch][4], s[batch][4]; proofs_out[batch][192]. */
int zk_groth16_prove_batch(zk_ctx *ctx, const zk_params *p, size_t batch,
                           const uint64_t *a_evals, const uint64_t *b_evals, const uint64_t *c_evals, size_t n_constraints,
                           const uint64_t *input_assignment, size_t n_inputs,
                           const uint64_t *aux_assignment, size_t n_aux,
                           const uint8_t *a_aux_density, const uint8_t *b_input_density, const uint8_t *b_aux_density,
                           const uint64_t *r, const uint64_t *s, uint8_t *proofs_out);

/* ---- proving straight from the witness (SURVEY.md §8 f4: synthesis off the critical path) --------------
 * For a FIXED circuit the constraint matrices A, B, C are known after one synthesis pass (bellman's
 * KeypairAssembly records them as at/bt/ct during parameter generation).  Loaded once in CSR form, the device
 * evaluates <A_j,z>, <B_j,z>, <C_j,z> itself, so per proof only the assignment z = (inputs | aux) crosses PCIe
 * (0.64 MB instead of 2.6 MB for confidential_transfer) and ProvingAssignment::enforce's host arithmetic disappears.
 *   row_ptr[n_constraints + 1], col[nnz] (variable index: < n_inputs = input, else n_inputs + aux index),
 *   coeff[nnz][4] canonical Fr.  The `input_i * 0 = 0` rows are appended by the library; densities are derived. */
typedef struct zk_r1cs zk_r1cs;
int zk_r1cs_load(zk_ctx *ctx, size_t n_constraints, size_t n_inputs, size_t n_aux,
                 const uint32_t *a_row_ptr, const uint32_t *a_col, const uint64_t *a_coeff,
                 const uint32_t *b_row_ptr, const uint32_t *b_col, const uint64_t *b_coeff,
                 const uint32_t *c_row_ptr, const uint32_t *c_col, const uint64_t *c_coeff, zk_r1cs **out);
void zk_r1cs_free(zk_r1cs *r1cs);
int zk_groth16_prove_witness_batch(zk_ctx *ctx, const zk_params *p, const zk_r1cs *r1cs, size_t batch,
                                   const uint64_t *input_assignment, const uint64_t *aux_assignment,
                                   const uint64_t *r, const uint64_t *s, uint8_t *proofs_out);

/* ---- parameter generation (replaces bellman::groth16::generate_parameters) ---------------------------------------------
 * generate_parameters (bellman groth16 generator.rs; reference calls core/proofs/src/setup.rs:28,59 through
 * generate_random_parameters, which draws g1, g2, alpha, beta, gamma, delta, tau from the rng).
 * r1cs: the circuit's constraints (zk_r1cs_load; the `input_i * 0 = 0` rows are appended here as in bellman).
 * g1, g2: G1Uncompressed / G2Uncompressed, checked (on curve, r-torsion, not infinity).
 * tau..delta: canonical FrRepr.  out: resident parameters, ready to prove with, equal to what zk_params_load would give
 * for the bytes bellman's Parameters::write emits for the same inputs.
 * Errors: ZK_ERR_NOT_CANONICAL (a scalar >= r), ZK_ERR_UNEXPECTED_IDENTITY (gamma or delta = 0 as in bellman; also alpha = 0,
 * beta = 0, tau = 0 or tau^m = 1, whose points zk_params_load would reject; a generator at infinity), ZK_ERR_DECODE (a generator
 * off the curve or outside the subgroup), ZK_ERR_UNCONSTRAINED_VARIABLE, ZK_ERR_POLY_DEGREE_TOO_LARGE (domain above 2^28 or a
 * vector of 2^26 points or more), ZK_ERR_INVALID (r1cs on another device).  The device buffers that held the trapdoor or values
 * derived from it are cleared before the call returns. */
int zk_groth16_generate(zk_ctx *ctx, const zk_r1cs *r1cs, const uint8_t g1[96], const uint8_t g2[192],
                        const uint64_t alpha[4], const uint64_t beta[4], const uint64_t gamma[4],
                        const uint64_t delta[4], const uint64_t tau[4], zk_params **out);

/* ---- utilities / diagnostics ------------------------------------------------------------------ */
/* out[i] = scalars[i] * base (limb form in, limb form out); group 1 or 2; any 256-bit scalar.  Used to build synthetic
 * CRS / test vectors on the device (the batched fixed-base multiplication of zk_groth16_generate). */
int zk_scalar_mul_many(zk_ctx *ctx, int group, const uint64_t *base_limbs, const uint64_t *scalars, size_t n,
                       uint64_t *out_limbs);
/* element-wise field ops on host arrays (parity tests of the device arithmetic):
 * field 0 = Fq (6 limbs), 1 = Fr (4 limbs); op 0 mul, 1 add, 2 sub, 3 sqr, 4 inverse, 5 from_repr, 6 into_repr */
int zk_field_op(zk_ctx *ctx, int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out);
/* calibrates the modmul roofline: runs `iters` dependent-chain-free Montgomery products per thread
 * over blocks x threads threads, returns products per second (field 0 Fq, 1 Fr). */
int zk_bench_modmul(zk_ctx *ctx, int field, int blocks, int threads, int iters, double *modmul_per_s, double *ms);

/* Live timing of the dominant kernel (the MSM bucket accumulation) with CUDA events recorded on the
 * context's stream around each launch: enable, run the workload, read the summed duration and launch
 * count (bench.py's roofline block).  Disabled by default (no events are created). */
int zk_ctx_profile(zk_ctx *ctx, int enable);
int zk_ctx_profile_read(zk_ctx *ctx, double *total_ms, uint64_t *launches);
/* Work executed by the MSMs of this context (and of its prover lanes) since the last zk_ctx_profile call, counted on the device:
 * the number of bucket additions (= non-zero signed digits) in G1 and in G2, and how many of them were left to the XYZZ pass
 * (the others were done by batched-affine rounds).  bench.py turns them into executed Fq-modmul-equivalents for the rooflines:
 * an XYZZ mixed addition = 10 products in the base field, a batched-affine addition = 6.4. */
int zk_ctx_profile_counts(zk_ctx *ctx, uint64_t *g1_additions, uint64_t *g2_additions, uint64_t *g1_xyzz, uint64_t *g2_xyzz);

/* ---- Groth16 verification (SURVEY.md §8 f2: the step after the proving path) ----------------------------------
 * zk_pvk: bellman_verifier::PreparedVerifyingKey<Bls12> resident on the device — e(alpha_g1, beta_g2), the Miller-loop
 * line coefficients of -gamma_g2 and -delta_g2, ic, and a fixed-base table of ic[1..] for the public-input sums. */
typedef struct zk_pvk zk_pvk;
/* PreparedVerifyingKey::read (core/bellman-verifier/src/lib.rs:204-245): the bytes zface ships as conf_vk.dat /
 * anony_vk.dat and modules/zk-system keeps in storage.  ic points are checked (on curve, subgroup, not infinity). */
int zk_pvk_load(zk_ctx *ctx, const uint8_t *pvk_bytes, size_t len, zk_pvk **out);
/* prepare_verifying_key(&vk) (core/bellman-verifier/src/verifier.rs:15-30) computed on the device from the VerifyingKey
 * encoding (alpha_g1 | beta_g1 | beta_g2 | gamma_g2 | delta_g1 | delta_g2 | u32 n | ic) — the head of Parameters::write,
 * so a proving-key buffer can be passed as is (trailing bytes are ignored). */
int zk_pvk_prepare(zk_ctx *ctx, const uint8_t *vk_bytes, size_t len, zk_pvk **out);
/* PreparedVerifyingKey::write (lib.rs:183-202): zk_pvk_size bytes, byte-identical to the reference's file */
size_t zk_pvk_size(const zk_pvk *k);
int zk_pvk_write(const zk_pvk *k, uint8_t *out);
size_t zk_pvk_num_inputs(const zk_pvk *k);      /* ic.len() - 1 */
void zk_pvk_free(zk_pvk *k);
/* Proof::read (lib.rs:67-108) + verify_proof (verifier.rs:32-63) for n proofs against one key.
 * proofs: n * 192 bytes (Proof::write); inputs: n * n_inputs canonical Fr (4 LE u64 each, FrRepr);
 * verdicts[i]: 1 = Ok(true), 0 = Ok(false), 2 = Proof::read failed with InvalidData (bad flags, x >= q, not on curve,
 * not in the subgroup), 3 = Proof::read failed with PointInfinity.  Returns ZK_ERR_MALFORMED_VK when
 * n_inputs + 1 != ic.len(), ZK_ERR_NOT_CANONICAL when an input is >= r. */
int zk_groth16_verify_batch(zk_ctx *ctx, const zk_pvk *k, size_t n, const uint8_t *proofs, const uint64_t *inputs,
                            size_t n_inputs, uint8_t *verdicts);
/* same with device pointers; asynchronous on the context's stream (zk_ctx_sync reports a pending ZK_ERR_NOT_CANONICAL) */
int zk_groth16_verify_batch_device(zk_ctx *ctx, const zk_pvk *k, size_t n, const uint8_t *d_proofs, const uint64_t *d_inputs,
                                   size_t n_inputs, uint8_t *d_verdicts);
/* Engine::pairing (core/pairing/src/lib.rs:108-115, bls12_381/mod.rs:40-160) for n pairs of checked G1Uncompressed /
 * G2Uncompressed encodings; out: n * 576 bytes in Fq12::write order (fq12.rs:29-45). */
int zk_pairing_batch(zk_ctx *ctx, size_t n, const uint8_t *g1, const uint8_t *g2, uint8_t *out);

#ifdef __cplusplus
}
#endif
#endif /* ZKB200_H */
