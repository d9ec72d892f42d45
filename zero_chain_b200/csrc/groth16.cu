// Groth16 prover orchestration on the device: CRS loading and create_proof below synthesis.
//
// Replaces upstream bellman 0.1.0 (un-vendored; SURVEY.md §3.2/§3.3):
//   groth16::Parameters::read(reader, checked)   <- core/proofs/src/confidential.rs:95-103
//   groth16::create_proof(circuit, params, r, s) <- core/proofs/src/confidential.rs:149 (via create_random_proof)
// and emits Proof::write bytes (core/bellman-verifier/src/lib.rs:55-65).
//
// B200-first restructuring of create_proof (same group elements, fewer serial scalar multiplications):
// the blinding terms are folded into the MSMs by appending vk points to the query vectors at load time,
//     a'    = a    ++ [alpha_g1, delta_g1]   scalars  inputs ++ aux|A-density ++ [1, r]   -> g_a
//     b_g1' = b_g1 ++ [beta_g1,  delta_g1]   scalars  inputs|B ++ aux|B       ++ [1, s]   -> g_b1
//     b_g2' = b_g2 ++ [beta_g2,  delta_g2]   scalars  (same)                              -> g_b
//     h'    = h    ++ [delta_g1]             scalars  h coefficients ++ [-(r s)]          -> H - rs*delta
//   g_c = s*g_a + r*g_b1 + (H - rs*delta_g1) + L
// which equals bellman's  delta*rs + alpha*s + beta*r + A*s + B1*r + H + L.  A whole batch of proofs
// shares every launch: NTTs are batched (grid.y) and each MSM uses one window set per proof.
#define ZK_SEMI_HOT 1   // Fq product inlined into the (noinline) point operations: shorter dependent chains in k_scale_points / k_finish_proofs
#include <stdlib.h>
#include "internal.h"
#include "codec.cuh"
#include "curve_coop.cuh"

struct zk_params {
    int device = 0;
    uint64_t n_ic = 0, n_h = 0, n_l = 0, n_a = 0, n_b1 = 0, n_b2 = 0;
    zk_bases *h = nullptr, *l = nullptr, *a = nullptr, *b1 = nullptr, *b2 = nullptr;   // extended vectors (see above)
    // the VerifyingKey part, kept so that Parameters::write and `params.vk` (core/proofs/src/setup.rs:31) can be served from the
    // resident CRS: G1 = alpha_g1, beta_g1, delta_g1, ic[n_ic]; G2 = beta_g2, gamma_g2, delta_g2 (affine, Montgomery)
    G1Affine *d_vk1 = nullptr;
    G2Affine *d_vk2 = nullptr;
    bool subgroup_checked = false;     // every point passed the r-torsion test at load time (checked load, or a cache written by one)
};

// The fixed constraint system of one circuit, resident on the device in CSR form (SURVEY.md §8 f4).
struct zk_r1cs {
    int device = 0;
    size_t n_c = 0, n_in = 0, n_aux = 0, nnz[3] = {0, 0, 0};
    uint32_t *d_row_ptr[3] = {nullptr, nullptr, nullptr}, *d_col[3] = {nullptr, nullptr, nullptr};
    void *d_coeff[3] = {nullptr, nullptr, nullptr};
    std::vector<uint8_t> a_aux_density, b_input_density, b_aux_density;     // DensityTracker bits, derived from A and B
};

static uint32_t rd_u32be(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
static void wr_u32be(uint8_t *p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }

extern "C" void zk_params_free(zk_params *p) {
    if (!p) return;
    zk_bases_free(p->h); zk_bases_free(p->l); zk_bases_free(p->a); zk_bases_free(p->b1); zk_bases_free(p->b2);
    cudaSetDevice(p->device);
    if (p->d_vk1) cudaFree(p->d_vk1);
    if (p->d_vk2) cudaFree(p->d_vk2);
    delete p;
}
extern "C" int zk_params_counts(const zk_params *p, uint64_t c[6]) {
    if (!p || !c) { zk_set_error("zk_params_counts: NULL argument"); return ZK_ERR_INVALID; }
    c[0] = p->n_ic; c[1] = p->n_h; c[2] = p->n_l; c[3] = p->n_a; c[4] = p->n_b1; c[5] = p->n_b2;
    return ZK_OK;
}

static const size_t VK_FIXED = 96 + 96 + 192 + 192 + 96 + 192;   // alpha_g1 | beta_g1 | beta_g2 | gamma_g2 | delta_g1 | delta_g2
static const uint32_t CRS_POINT_LIMIT = 1u << 26;                // zk_bases_from_device accepts < 2^27 bases

// Device-side layout of a decoded CRS before the tables are built: the five EXTENDED query vectors and the vk points.
// g1 = h' | l | a' | b_g1' | vk1 (alpha, beta_g1, delta, ic...),  g2 = b_g2' | vk2 (beta_g2, gamma_g2, delta_g2)
struct CrsLayout {
    size_t cnt[6];                               // ic, h, l, a, b_g1, b_g2 as stored in the stream
    size_t n_h, n_l, n_a, n_b1, n_b2, n_vk1;     // extended lengths
    size_t o_h, o_l, o_a, o_b1, o_vk1;           // offsets (points) inside g1
    size_t g1_total, g2_total;
    explicit CrsLayout(const size_t c[6]) {
        for (int k = 0; k < 6; k++) cnt[k] = c[k];
        n_h = c[1] + 1; n_l = c[2]; n_a = c[3] + 2; n_b1 = c[4] + 2; n_b2 = c[5] + 2; n_vk1 = 3 + c[0];
        o_h = 0; o_l = o_h + n_h; o_a = o_l + n_l; o_b1 = o_a + n_a; o_vk1 = o_b1 + n_b1;
        g1_total = o_vk1 + n_vk1; g2_total = n_b2 + 3;
    }
};
// tables + handle from decoded device arrays (shared by the byte-stream loader and the decoded-CRS cache)
static int params_from_device(zk_ctx *ctx, const CrsLayout &L, const G1Affine *g1, const G2Affine *g2, zk_params **out) {
    zk_params *p = new zk_params();
    p->device = ctx->device;
    p->n_ic = L.cnt[0]; p->n_h = L.cnt[1]; p->n_l = L.cnt[2]; p->n_a = L.cnt[3]; p->n_b1 = L.cnt[4]; p->n_b2 = L.cnt[5];
    int r = ZK_OK;
    if (cudaMalloc(&p->d_vk1, L.n_vk1 * sizeof(G1Affine)) != cudaSuccess || cudaMalloc(&p->d_vk2, 3 * sizeof(G2Affine)) != cudaSuccess) {
        zk_set_error("cudaMalloc (verifying key) failed"); zk_params_free(p); return ZK_ERR_CUDA;
    }
    cudaMemcpyAsync(p->d_vk1, g1 + L.o_vk1, L.n_vk1 * sizeof(G1Affine), cudaMemcpyDeviceToDevice, ctx->stream);
    cudaMemcpyAsync(p->d_vk2, g2 + L.n_b2, 3 * sizeof(G2Affine), cudaMemcpyDeviceToDevice, ctx->stream);
    // window tables (built once; the CRS is fixed)
    int wb_h = 0;
#ifdef ZK_EXPERIMENTS
    if (const char *e = getenv("ZK_WB_H")) wb_h = atoi(e);          // experiment knob: window bits of the H-query tables (0 = automatic)
#endif
    if ((r = zk_bases_from_device(ctx, 1, g1 + L.o_h, L.n_h, wb_h, 1, &p->h)) || (r = zk_bases_from_device(ctx, 1, g1 + L.o_l, L.n_l, 0, 1, &p->l)) ||
        (r = zk_bases_from_device(ctx, 1, g1 + L.o_a, L.n_a, 0, 1, &p->a)) || (r = zk_bases_from_device(ctx, 1, g1 + L.o_b1, L.n_b1, 0, 1, &p->b1)) ||
        (r = zk_bases_from_device(ctx, 2, g2, L.n_b2, 0, 1, &p->b2))) {
        zk_params_free(p);
        return r;
    }
    *out = p;
    return ZK_OK;
}
// host: walk the grammar (SURVEY.md §3.3) to find the vectors; no arithmetic here
static int params_walk(const uint8_t *buf, size_t len, size_t voff[6], size_t vcnt[6]) {
    size_t off = VK_FIXED;
    const size_t vsz[6] = {96, 96, 96, 96, 96, 192};
    for (int k = 0; k < 6; k++) {
        if (off + 4 > len) { zk_set_error("Parameters stream truncated (length prefix %d)", k); return ZK_ERR_IO; }
        vcnt[k] = rd_u32be(buf + off); off += 4;
        voff[k] = off;
        if (vcnt[k] > (len - off) / vsz[k]) { zk_set_error("Parameters stream truncated (vector %d: %zu points)", k, vcnt[k]); return ZK_ERR_IO; }
        off += vcnt[k] * vsz[k];
    }
    if (vcnt[1] == 0 || vcnt[2] == 0 || vcnt[3] == 0 || vcnt[4] == 0 || vcnt[5] == 0) { zk_set_error("empty query vector in Parameters"); return ZK_ERR_IO; }
    for (int k = 0; k < 6; k++) if (vcnt[k] >= CRS_POINT_LIMIT) { zk_set_error("Parameters vector %d too long (%zu points)", k, vcnt[k]); return ZK_ERR_IO; }
    return ZK_OK;
}
// decode the stream into stage_b (G1) / stage_c (G2) in the CrsLayout order
static int params_decode(zk_ctx *ctx, const uint8_t *buf, size_t len, int checked, const size_t voff[6], const CrsLayout &L) {
    ZK_TRY(ctx->stage_a.reserve(len));
    ZK_CUDA(cudaMemcpyAsync(ctx->stage_a.p, buf, len, cudaMemcpyHostToDevice, ctx->stream));
    const uint8_t *d = ctx->stage_a.as<uint8_t>();
    ZK_TRY(ctx->stage_b.reserve((L.g1_total + 8) * sizeof(G1Affine)));
    ZK_TRY(ctx->stage_c.reserve((L.g2_total + 8) * sizeof(G2Affine)));
    G1Affine *g1 = ctx->stage_b.as<G1Affine>();
    G1Affine *dh = g1 + L.o_h, *dl = g1 + L.o_l, *da = g1 + L.o_a, *db1 = g1 + L.o_b1, *dvk = g1 + L.o_vk1;
    G2Affine *db2 = ctx->stage_c.as<G2Affine>(), *dvk2 = db2 + L.n_b2;
    int *err = ctx->d_err + 1;
    auto dec1 = [&](size_t boff, size_t n, G1Affine *dst, int reject_inf) {
        if (n) zkcodec::k_decode_uncompressed<Fq><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d + boff, n, checked, reject_inf, dst, err);
    };
    auto dec2 = [&](size_t boff, size_t n, G2Affine *dst, int reject_inf) {
        if (n) zkcodec::k_decode_uncompressed<Fq2><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d + boff, n, checked, reject_inf, dst, err);
    };
    const size_t *vcnt = L.cnt;
    // vk: alpha_g1 @0, beta_g1 @96, beta_g2 @192, gamma_g2 @384, delta_g1 @576, delta_g2 @672
    dec1(voff[1], vcnt[1], dh, 1);          dec1(576, 1, dh + vcnt[1], 1);                                  // h ++ [delta_g1]
    dec1(voff[2], vcnt[2], dl, 1);
    dec1(voff[3], vcnt[3], da, 1);          dec1(0, 1, da + vcnt[3], 1);    dec1(576, 1, da + vcnt[3] + 1, 1);   // a ++ [alpha, delta]
    dec1(voff[4], vcnt[4], db1, 1);         dec1(96, 1, db1 + vcnt[4], 1);  dec1(576, 1, db1 + vcnt[4] + 1, 1);  // b_g1 ++ [beta_g1, delta]
    dec2(voff[5], vcnt[5], db2, 1);         dec2(192, 1, db2 + vcnt[5], 1); dec2(672, 1, db2 + vcnt[5] + 1, 1);  // b_g2 ++ [beta_g2, delta_g2]
    // verifying key as it stands in the stream (already validated above where it overlaps): alpha, beta_g1, delta, ic | beta_g2, gamma_g2, delta_g2
    dec1(0, 1, dvk, 1); dec1(96, 1, dvk + 1, 1); dec1(576, 1, dvk + 2, 1);
    dec1(voff[0], vcnt[0], dvk + 3, 0);                                                                   // ic: infinity allowed (bellman reads it as is)
    dec2(192, 1, dvk2, 1); dec2(384, 1, dvk2 + 1, 0); dec2(672, 1, dvk2 + 2, 1);                           // gamma_g2: not used by the prover
    ZK_CUDA(cudaGetLastError());
    return zk_check_err_flag(ctx);
}

extern "C" int zk_params_load(zk_ctx *ctx, const uint8_t *buf, size_t len, int checked, zk_params **out) {
    if (!ctx || !buf || !out) { zk_set_error("zk_params_load: NULL argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    size_t voff[6], vcnt[6];
    ZK_TRY(params_walk(buf, len, voff, vcnt));
    CrsLayout L(vcnt);
    ZK_TRY(params_decode(ctx, buf, len, checked, voff, L));
    ZK_TRY(params_from_device(ctx, L, ctx->stage_b.as<G1Affine>(), ctx->stage_c.as<G2Affine>(), out));
    (*out)->subgroup_checked = checked != 0;
    return ZK_OK;
}

// ---- Parameters::write from the resident CRS --------------------------------------------------------------------------
// (bellman groth16 Parameters::write: vk.write, then h, l, a, b_g1, b_g2 each as u32 BE length + uncompressed points; reference call
// core/proofs/src/confidential.rs:83 `self.proving_key.write(&mut &mut v_pk)`.)  The device holds canonical affine points in
// Montgomery form, and the Uncompressed encoding of a point is unique, so decode -> encode reproduces the input stream byte for byte.
extern "C" size_t zk_params_size(const zk_params *p) {
    if (!p) return 0;
    return VK_FIXED + 4 + 96 * p->n_ic + 4 + 96 * p->n_h + 4 + 96 * p->n_l + 4 + 96 * p->n_a + 4 + 96 * p->n_b1 + 4 + 192 * p->n_b2;
}
extern "C" size_t zk_params_vk_size(const zk_params *p) { return p ? VK_FIXED + 4 + 96 * p->n_ic : 0; }
static int params_write_impl(zk_ctx *ctx, const zk_params *p, uint8_t *out, bool vk_only) {
    if (!ctx || !p || !out) { zk_set_error("zk_params_write: NULL argument"); return ZK_ERR_INVALID; }
    if (p->device != ctx->device) { zk_set_error("params live on device %d, context on %d", p->device, ctx->device); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    const size_t total = vk_only ? zk_params_vk_size(p) : zk_params_size(p);
    ZK_TRY(ctx->stage_a.reserve(total));
    uint8_t *d = ctx->stage_a.as<uint8_t>();
    cudaStream_t st = ctx->stream;
    auto enc1 = [&](const G1Affine *src, size_t n, size_t boff) {
        if (n) zkcodec::k_encode_affine<Fq><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(src, n, d + boff);
    };
    auto enc2 = [&](const G2Affine *src, size_t n, size_t boff) {
        if (n) zkcodec::k_encode_affine<Fq2><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(src, n, d + boff);
    };
    enc1(p->d_vk1, 1, 0); enc1(p->d_vk1 + 1, 1, 96); enc2(p->d_vk2, 1, 192); enc2(p->d_vk2 + 1, 1, 384); enc1(p->d_vk1 + 2, 1, 576); enc2(p->d_vk2 + 2, 1, 672);
    size_t off = VK_FIXED, pre[6];
    pre[0] = off; off += 4; enc1(p->d_vk1 + 3, p->n_ic, off); off += 96 * p->n_ic;
    if (!vk_only) {
        pre[1] = off; off += 4; enc1((const G1Affine *)p->h->d_tbl, p->n_h, off); off += 96 * p->n_h;
        pre[2] = off; off += 4; enc1((const G1Affine *)p->l->d_tbl, p->n_l, off); off += 96 * p->n_l;
        pre[3] = off; off += 4; enc1((const G1Affine *)p->a->d_tbl, p->n_a, off); off += 96 * p->n_a;
        pre[4] = off; off += 4; enc1((const G1Affine *)p->b1->d_tbl, p->n_b1, off); off += 96 * p->n_b1;
        pre[5] = off; off += 4; enc2((const G2Affine *)p->b2->d_tbl, p->n_b2, off); off += 192 * p->n_b2;
    }
    ZK_CUDA(cudaGetLastError());
    ZK_CUDA(cudaMemcpyAsync(out, d, total, cudaMemcpyDeviceToHost, st));
    ZK_CUDA(cudaStreamSynchronize(st));
    const uint64_t cnt[6] = {p->n_ic, p->n_h, p->n_l, p->n_a, p->n_b1, p->n_b2};
    for (int k = 0; k < (vk_only ? 1 : 6); k++) wr_u32be(out + pre[k], (uint32_t)cnt[k]);
    return ZK_OK;
}
extern "C" int zk_params_write(zk_ctx *ctx, const zk_params *p, uint8_t *out) { return params_write_impl(ctx, p, out, false); }
extern "C" int zk_params_write_vk(zk_ctx *ctx, const zk_params *p, uint8_t *out) { return params_write_impl(ctx, p, out, true); }

// ---- decoded-CRS cache on disk (SURVEY.md §8 f1; the "FIX: too heavy" read at core/proofs/src/crypto_components.rs:320) --------------
// First load of a proving key: zk_params_load(checked) + the decoded Montgomery points written to `cache_path`.  Later loads of the
// SAME bytes (SHA-256 guard over the whole stream) upload the decoded points directly: no decoding, no on-curve / subgroup tests.
namespace {
struct Sha256 {
    uint32_t h[8]; uint8_t blk[64]; size_t fill = 0; uint64_t total = 0;
    Sha256() { static const uint32_t iv[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u}; memcpy(h, iv, 32); }
    static uint32_t ror(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
    void block(const uint8_t *p) {
        static const uint32_t K[64] = {
            0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u, 0xd807aa98u, 0x12835b01u, 0x243185beu, 0x550c7dc3u,
            0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u, 0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu, 0x2de92c6fu, 0x4a7484aau, 0x5cb0a9dcu, 0x76f988dau,
            0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u, 0x06ca6351u, 0x14292967u, 0x27b70a85u, 0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u,
            0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u, 0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u, 0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u,
            0x19a4c116u, 0x1e376c08u, 0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu, 0x682e6ff3u, 0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u,
            0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u};
        uint32_t w[64];
        for (int i = 0; i < 16; i++) w[i] = rd_u32be(p + 4 * i);
        for (int i = 16; i < 64; i++) {
            uint32_t s0 = ror(w[i - 15], 7) ^ ror(w[i - 15], 18) ^ (w[i - 15] >> 3), s1 = ror(w[i - 2], 17) ^ ror(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
        for (int i = 0; i < 64; i++) {
            uint32_t t1 = hh + (ror(e, 6) ^ ror(e, 11) ^ ror(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
            uint32_t t2 = (ror(a, 2) ^ ror(a, 13) ^ ror(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
            hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    void update(const uint8_t *p, size_t n) {
        total += n;
        if (fill) { size_t k = 64 - fill < n ? 64 - fill : n; memcpy(blk + fill, p, k); fill += k; p += k; n -= k; if (fill == 64) { block(blk); fill = 0; } }
        for (; n >= 64; p += 64, n -= 64) block(p);
        if (n) { memcpy(blk, p, n); fill = n; }
    }
    void finish(uint8_t out[32]) {
        uint64_t bits = total * 8;
        uint8_t pad[72] = {0x80};
        size_t k = (fill < 56 ? 56 : 120) - fill;
        update(pad, k);
        uint8_t lenb[8];
        for (int i = 0; i < 8; i++) lenb[i] = (uint8_t)(bits >> (56 - 8 * i));
        update(lenb, 8);
        for (int i = 0; i < 8; i++) wr_u32be(out + 4 * i, h[i]);
    }
};
struct CacheHeader {
    char magic[8];              // "ZKB2CRS1"
    uint64_t pk_len;
    uint8_t sha[32];
    uint64_t cnt[6];
    uint64_t g1_points, g2_points;
    uint8_t body_sha[32];       // SHA-256 of the decoded points that follow: a hit skips every check, so the body must be what was written
};
}  // namespace
extern "C" int zk_params_load_cached(zk_ctx *ctx, const uint8_t *buf, size_t len, const char *cache_path, int *cache_hit, zk_params **out) {
    if (!ctx || !buf || !out || !cache_path) { zk_set_error("zk_params_load_cached: NULL argument"); return ZK_ERR_INVALID; }
    if (cache_hit) *cache_hit = 0;
    ZK_TRY(zk_use_device(ctx));
    size_t voff[6], vcnt[6];
    ZK_TRY(params_walk(buf, len, voff, vcnt));
    CrsLayout L(vcnt);
    CacheHeader want;
    memset(&want, 0, sizeof(want));
    memcpy(want.magic, "ZKB2CRS1", 8);
    want.pk_len = len;
    { Sha256 s; s.update(buf, len); s.finish(want.sha); }
    for (int k = 0; k < 6; k++) want.cnt[k] = vcnt[k];
    want.g1_points = L.g1_total; want.g2_points = L.g2_total;
    const size_t b1 = L.g1_total * sizeof(G1Affine), b2 = L.g2_total * sizeof(G2Affine);
    if (FILE *f = fopen(cache_path, "rb")) {
        CacheHeader got;
        std::vector<uint8_t> body;
        bool ok = fread(&got, sizeof(got), 1, f) == 1 && memcmp(&got, &want, offsetof(CacheHeader, body_sha)) == 0;
        if (ok) { body.resize(b1 + b2); ok = fread(body.data(), 1, b1 + b2, f) == b1 + b2 && fgetc(f) == EOF; }
        fclose(f);
        if (ok) { uint8_t h[32]; Sha256 sh; sh.update(body.data(), body.size()); sh.finish(h); ok = memcmp(h, got.body_sha, 32) == 0; }
        if (ok) {
            ZK_TRY(ctx->stage_b.reserve(b1 + 8 * sizeof(G1Affine)));
            ZK_TRY(ctx->stage_c.reserve(b2 + 8 * sizeof(G2Affine)));
            ZK_CUDA(cudaMemcpyAsync(ctx->stage_b.p, body.data(), b1, cudaMemcpyHostToDevice, ctx->stream));
            ZK_CUDA(cudaMemcpyAsync(ctx->stage_c.p, body.data() + b1, b2, cudaMemcpyHostToDevice, ctx->stream));
            ZK_CUDA(cudaStreamSynchronize(ctx->stream));
            if (cache_hit) *cache_hit = 1;
            ZK_TRY(params_from_device(ctx, L, ctx->stage_b.as<G1Affine>(), ctx->stage_c.as<G2Affine>(), out));
            (*out)->subgroup_checked = true;       // the cache is only ever written after a checked load, and its body is hash-guarded
            return ZK_OK;
        }
    }
    // miss (absent, other key, truncated): the full checked load, then the cache is (re)written
    ZK_TRY(params_decode(ctx, buf, len, 1, voff, L));
    std::vector<uint8_t> body(b1 + b2);
    ZK_CUDA(cudaMemcpyAsync(body.data(), ctx->stage_b.p, b1, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaMemcpyAsync(body.data() + b1, ctx->stage_c.p, b2, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    ZK_TRY(params_from_device(ctx, L, ctx->stage_b.as<G1Affine>(), ctx->stage_c.as<G2Affine>(), out));
    (*out)->subgroup_checked = true;
    { Sha256 sh; sh.update(body.data(), body.size()); sh.finish(want.body_sha); }
    std::string tmp = std::string(cache_path) + ".tmp";
    if (FILE *f = fopen(tmp.c_str(), "wb")) {           // a cache that cannot be written is not an error of the load
        bool ok = fwrite(&want, sizeof(want), 1, f) == 1 && fwrite(body.data(), 1, body.size(), f) == body.size();
        ok = (fclose(f) == 0) && ok;
        if (ok) rename(tmp.c_str(), cache_path); else remove(tmp.c_str());
    }
    return ZK_OK;
}

// ---- prove -----------------------------------------------------------------------------------------------
namespace {
// out[b][k] = src[b][idx[k]]  (32-byte elements)
__global__ void k_gather32(const uint4 *__restrict__ src, size_t src_stride, const uint32_t *__restrict__ idx, size_t n_idx,
                           uint4 *__restrict__ dst, size_t dst_stride, size_t dst_off) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (k >= n_idx) return;
    const uint4 *s = src + (b * src_stride + idx[k]) * 2;
    uint4 *d = dst + (b * dst_stride + dst_off + k) * 2;
    d[0] = s[0]; d[1] = s[1];
}
// dst[b][dst_off + j] = terms[b][sel_j]
__global__ void k_put_terms(const uint4 *__restrict__ terms, int sel0, int sel1, int n_sel, uint4 *__restrict__ dst, size_t dst_stride,
                            size_t dst_off, size_t batch) {
    size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    for (int j = 0; j < n_sel; j++) {
        int sel = j ? sel1 : sel0;
        const uint4 *s = terms + (b * 4 + sel) * 2;
        uint4 *d = dst + (b * dst_stride + dst_off + j) * 2;
        d[0] = s[0]; d[1] = s[1];
    }
}
// block per (proof, j): T[b][j] = (j == 0 ? s : r) * (j == 0 ? g_a : g_b1).  A 255-bit double-and-add on one thread is ~380
// dependent point operations; here thread 0 runs the doubling chain 2^i P into shared memory (the only serial part) and the
// block then sums the selected powers: 4 per thread, then a 6-level tree — about 2.5x less latency for the same group element.
constexpr int SCALE_T = 64;
// `glv` != 0 (the CRS was loaded CHECKED, so g_a and g_b1 lie in the r-torsion): k P is split with the curve endomorphism
// phi(x, y) = (beta x, y) = -[u^2] P (u the BLS parameter; the identity the subgroup test of codec.cuh uses, exact on G1):
// k = k1 u^2 + k0 by plain division (k0, k1 < 2^128), so k P = k0 P - k1 phi(P) and phi(2^i P) = 2^i phi(P): the doubling chain
// is 127 steps instead of 254.  Without the guarantee (unchecked load) the plain 254-step chain is used: same group element either way.
__global__ void __launch_bounds__(SCALE_T) k_scale_points(const G1XYZZ *__restrict__ ga, const G1XYZZ *__restrict__ gb1, const uint32_t *__restrict__ terms,
                                                          size_t batch, int j, int glv, G1XYZZ *__restrict__ T) {
    __shared__ G1XYZZ pw[255];                                                   // 2^i P, i <= 254; reused for the tree (47.8 KB)
    __shared__ uint32_t kk[2][4];                                                // glv: k0, k1
    const size_t b = blockIdx.x, id = 2 * b + j;                                 // one launch per product kind j (each on the lane that made its point)
    const int t = threadIdx.x;
    const uint32_t *k = terms + (b * 4 + (j ? 1 : 2)) * 8;                       // j=0: s, j=1: r
    int top = -1;
    for (int i = 7; i >= 0 && top < 0; i--) if (k[i]) top = 32 * i + 31 - __clz(k[i]);
    if (top > 254) top = 254;          // a non-canonical r / s (>= 2^255) is reported through the error flag by k_blinding_terms; stay inside pw[]
    if (glv && top > 127) top = 127;   // quotient and remainder are below 2^128 (u^2 > 2^127, k < 2^255)
    if (t < 32) {                                                               // warp 0: the doubling chain, three cooperative stages per doubling
        G1XYZZ d = j ? gb1[b] : ga[b];
        if (t == 0) pw[0] = d;
        for (int i = 1; i <= top; i++) { zkcoop::dbl(d); if (t == 0) pw[i] = d; }
    } else if (glv && t == 32) {                                                // meanwhile, on the other warp: k = k1 * u^2 + k0 by shift-and-subtract
        const uint32_t dv[4] = {0x00000000u, 0x00000001u, 0x0001a402u, 0xac45a401u};        // u^2 = 0xd201000000010000^2
        uint32_t rem[5] = {0, 0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
        for (int i = 254; i >= 0; i--) {
            for (int w = 4; w > 0; w--) rem[w] = (rem[w] << 1) | (rem[w - 1] >> 31);
            rem[0] = (rem[0] << 1) | ((k[i >> 5] >> (i & 31)) & 1);
            bool ge = rem[4] != 0;
            if (!ge) { ge = true; for (int w = 3; w >= 0; w--) { if (rem[w] != dv[w]) { ge = rem[w] > dv[w]; break; } } }
            if (ge) {
                uint64_t br = 0;
                for (int w = 0; w < 4; w++) { uint64_t x = (uint64_t)rem[w] - dv[w] - br; rem[w] = (uint32_t)x; br = (x >> 63) & 1; }
                rem[4] -= (uint32_t)br;
                if (i < 128) q[i >> 5] |= 1u << (i & 31);
            }
        }
        for (int w = 0; w < 4; w++) { kk[0][w] = rem[w]; kk[1][w] = q[w]; }
    }
    __syncthreads();
    G1XYZZ acc = G1XYZZ::inf();
    if (!glv) {
        for (int i = 4 * t; i < 4 * t + 4 && i <= top; i++)
            if ((k[i >> 5] >> (i & 31)) & 1) acc.add(pw[i]);
    } else {                                                                    // threads 0..31: bits of k0 on 2^i P; 32..63: bits of k1 on -phi(2^i P)
        const int half = t >> 5, i0 = 4 * (t & 31);
        const uint32_t beta_w[12] = ZK_ENDO_BETA_INIT;
        Fq beta; for (int w = 0; w < 12; w++) beta.l[w] = beta_w[w];
        for (int i = i0; i < i0 + 4 && i <= top; i++)
            if ((kk[half][i >> 5] >> (i & 31)) & 1) {
                G1XYZZ p = pw[i];
                if (half) { p.x = p.x * beta; p.y = p.y.neg(); }
                acc.add(p);
            }
    }
    __syncthreads();                                                             // every thread is done reading the powers
    G1XYZZ *part = pw;
    part[t] = acc;
    __syncthreads();
    for (int stride = SCALE_T / 2; stride > 0; stride >>= 1) {
        if (t < stride) { G1XYZZ a = part[t]; a.add(part[t + stride]); part[t] = a; }
        __syncthreads();
    }
    if (t == 0) T[id] = part[0];
}
// block of three warps per 32 proofs, one warp per proof element, so that the three affine conversions (a field inversion each) of a
// proof run side by side: warp 0 encodes A, warp 1 B (G2), warp 2 forms g_c = T0 + T1 + H' + L and encodes it.  Proof::write layout:
// compressed a | b | c.
__global__ void __launch_bounds__(96) k_finish_proofs(const G1XYZZ *__restrict__ ga, const G2XYZZ *__restrict__ gb, const G1XYZZ *__restrict__ T,
                                                      const G1XYZZ *__restrict__ H, const G1XYZZ *__restrict__ L, size_t batch, uint8_t *__restrict__ out) {
    const size_t b = (size_t)blockIdx.x * 32 + (threadIdx.x & 31);
    const int which = threadIdx.x >> 5;
    if (b >= batch) return;
    uint8_t *o = out + b * 192;
    if (which == 0) zkcodec::encode_point(o, ga[b].to_affine(), true);
    else if (which == 1) zkcodec::encode_point(o + 48, gb[b].to_affine(), true);
    else {
        G1XYZZ c = T[2 * b];
        c.add(T[2 * b + 1]); c.add(H[b]); c.add(L[b]);
        zkcodec::encode_point(o + 144, c.to_affine(), true);
    }
}
}  // namespace

// The four inter-lane events of one prove call.  If the call fails after the auxiliary lanes have been started, the lanes are
// drained (their kernels still read g_scal2 / g_scal3, which the next call would overwrite) and their error flags cleared,
// keeping the error text of the failure that caused the exit.
namespace {
struct LaneEvents {
    cudaEvent_t b = nullptr, g2 = nullptr, a = nullptr, l3 = nullptr, l4 = nullptr;
    zk_ctx *lane2 = nullptr, *lane3 = nullptr, *lane4 = nullptr;
    bool lanes_started = false, completed = false;
    int create() {
        for (cudaEvent_t *e : {&b, &g2, &a, &l3, &l4}) ZK_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        return ZK_OK;
    }
    ~LaneEvents() {
        if (lanes_started && !completed) {
            std::string keep = zk_last_error();
            for (zk_ctx *l : {lane2, lane3, lane4}) { cudaStreamSynchronize(l->stream); zk_check_err_flag(l); }
            zk_set_error("%s", keep.c_str());
        }
        for (cudaEvent_t e : {b, g2, a, l3, l4}) if (e) cudaEventDestroy(e);
    }
};
}  // namespace

// batches larger than PROVE_CHUNK are processed in slices (device workspace and the 31-bit MSM entry index bound the slice)
static const size_t PROVE_CHUNK = 256;

static int prove_impl(zk_ctx *ctx, const zk_params *p, size_t batch,
                      const uint64_t *a_ev, const uint64_t *b_ev, const uint64_t *c_ev, size_t n_c,
                      const uint64_t *inputs, size_t n_in, const uint64_t *aux, size_t n_aux,
                      const uint8_t *a_aux_d, const uint8_t *b_in_d, const uint8_t *b_aux_d,
                      const uint64_t *r, const uint64_t *s, uint8_t *proofs_out, const zk_r1cs *r1cs = nullptr) {
    if (r1cs) {     // evaluations are computed on the device from the witness; densities come with the constraint system
        if (r1cs->n_in != n_in || r1cs->n_aux != n_aux) { zk_set_error("witness sizes do not match the constraint system"); return ZK_ERR_ASSIGNMENT_MISSING; }
        a_aux_d = r1cs->a_aux_density.data(); b_in_d = r1cs->b_input_density.data(); b_aux_d = r1cs->b_aux_density.data();
        n_c = r1cs->n_c + r1cs->n_in;
    }
    if (!ctx || !p || (!r1cs && (!a_ev || !b_ev || !c_ev)) || !inputs || !aux || !a_aux_d || !b_in_d || !b_aux_d || !r || !s || !proofs_out) {
        zk_set_error("zk_groth16_prove: NULL argument"); return ZK_ERR_INVALID;
    }
    if (batch == 0 || batch > PROVE_CHUNK || n_c == 0) { zk_set_error("zk_groth16_prove: bad batch / constraint count"); return ZK_ERR_INVALID; }
    if (p->device != ctx->device) { zk_set_error("params live on device %d, context on %d", p->device, ctx->device); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    cudaStream_t st = ctx->stream;
    // EvaluationDomain::from_coeffs
    unsigned log_m = 0; size_t m = 1;
    while (m < n_c) { m <<= 1; log_m++; if (log_m >= 32) { zk_set_error("PolynomialDegreeTooLarge"); return ZK_ERR_POLY_DEGREE_TOO_LARGE; } }
    // host-side density bookkeeping (DensityTracker::get_total_density and the query offsets of ParameterSource)
    std::vector<uint32_t> a_idx, bi_idx, ba_idx;
    for (size_t i = 0; i < n_aux; i++) { if (a_aux_d[i]) a_idx.push_back((uint32_t)i); if (b_aux_d[i]) ba_idx.push_back((uint32_t)i); }
    for (size_t i = 0; i < n_in; i++) if (b_in_d[i]) bi_idx.push_back((uint32_t)i);
    // ParameterSource::get_h / get_l / get_a / get_b_g1 / get_b_g2 size checks
    if (p->n_h != m - 1 || p->n_l != n_aux || p->n_a != n_in + a_idx.size() || p->n_b1 != bi_idx.size() + ba_idx.size() ||
        p->n_b2 != p->n_b1 || p->n_ic != n_in) {
        zk_set_error("witness shape does not match the CRS (h %llu vs %zu, l %llu vs %zu, a %llu vs %zu, b %llu vs %zu, ic %llu vs %zu)",
                     (unsigned long long)p->n_h, m - 1, (unsigned long long)p->n_l, n_aux, (unsigned long long)p->n_a, n_in + a_idx.size(),
                     (unsigned long long)p->n_b1, bi_idx.size() + ba_idx.size(), (unsigned long long)p->n_ic, n_in);
        return ZK_ERR_ASSIGNMENT_MISSING;
    }
    const size_t nH = p->n_h + 1, nA = p->n_a + 2, nB = p->n_b1 + 2;
    // ---- staging ----
    ZK_TRY(ctx->g_a.reserve(batch * 3 * m * 32));                    // a|b|c domains
    ZK_TRY(ctx->g_h.reserve(batch * m * 32));                        // quotient
    ZK_TRY(ctx->g_b.reserve(batch * n_c * 32));                      // raw evals staging
    ZK_TRY(ctx->g_c.reserve(batch * (n_in + n_aux) * 32 + 64));      // inputs | aux (canonical)
    size_t max_scal = nH; if (nA > max_scal) max_scal = nA; if (nB > max_scal) max_scal = nB;
    ZK_TRY(ctx->g_scal.reserve(batch * max_scal * 32));
    ZK_TRY(ctx->g_scal2.reserve(batch * nB * 32));
    if (!ctx->aux) { ZK_TRY(zk_ctx_create(ctx->device, nullptr, &ctx->aux)); ctx->aux->opts = ctx->opts; }      // second lane for the G2 MSM
    zk_ctx *lane2 = ctx->aux;
    ZK_TRY(ctx->g_scal3.reserve(batch * nA * 32));
    if (!ctx->aux2) { ZK_TRY(zk_ctx_create(ctx->device, nullptr, &ctx->aux2)); ctx->aux2->opts = ctx->opts; }    // third lane for the A and B1 MSMs
    zk_ctx *lane3 = ctx->aux2;
    if (!ctx->aux3) { ZK_TRY(zk_ctx_create(ctx->device, nullptr, &ctx->aux3)); ctx->aux3->opts = ctx->opts; }    // fourth lane for the B1 MSM
    zk_ctx *lane4 = ctx->aux3;
    auto rnd = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t misc_bytes = rnd(a_idx.size() * 4 + 4) + rnd(bi_idx.size() * 4 + 4) + rnd(ba_idx.size() * 4 + 4) + 2 * rnd(batch * 32) + rnd(batch * 128) +
                        4 * rnd(batch * sizeof(G1XYZZ)) + rnd(2 * batch * sizeof(G1XYZZ)) + rnd(batch * sizeof(G2XYZZ)) + rnd(batch * 192);
    ZK_TRY(ctx->g_misc.reserve(misc_bytes));
    uint8_t *mp = ctx->g_misc.as<uint8_t>();
    auto carve = [&](size_t bytes) { uint8_t *q = mp; mp += rnd(bytes); return q; };
    uint32_t *d_aidx = (uint32_t *)carve(a_idx.size() * 4 + 4), *d_biidx = (uint32_t *)carve(bi_idx.size() * 4 + 4), *d_baidx = (uint32_t *)carve(ba_idx.size() * 4 + 4);
    uint8_t *d_r = carve(batch * 32), *d_s = carve(batch * 32), *d_terms = carve(batch * 4 * 32);
    G1XYZZ *d_ga = (G1XYZZ *)carve(batch * sizeof(G1XYZZ)), *d_gb1 = (G1XYZZ *)carve(batch * sizeof(G1XYZZ));
    G1XYZZ *d_H = (G1XYZZ *)carve(batch * sizeof(G1XYZZ)), *d_L = (G1XYZZ *)carve(batch * sizeof(G1XYZZ)), *d_T = (G1XYZZ *)carve(2 * batch * sizeof(G1XYZZ));
    G2XYZZ *d_gb = (G2XYZZ *)carve(batch * sizeof(G2XYZZ));
    uint8_t *d_proofs = carve(batch * 192);
    if (a_idx.size()) ZK_CUDA(cudaMemcpyAsync(d_aidx, a_idx.data(), a_idx.size() * 4, cudaMemcpyHostToDevice, st));
    if (bi_idx.size()) ZK_CUDA(cudaMemcpyAsync(d_biidx, bi_idx.data(), bi_idx.size() * 4, cudaMemcpyHostToDevice, st));
    if (ba_idx.size()) ZK_CUDA(cudaMemcpyAsync(d_baidx, ba_idx.data(), ba_idx.size() * 4, cudaMemcpyHostToDevice, st));
    ZK_CUDA(cudaMemcpyAsync(d_r, r, batch * 32, cudaMemcpyHostToDevice, st));
    ZK_CUDA(cudaMemcpyAsync(d_s, s, batch * 32, cudaMemcpyHostToDevice, st));
    ZK_TRY(zk_fr_blinding_terms(ctx, d_r, d_s, batch, d_terms));
    // ---- h: 3 x (ifft, coset_fft), quotient, icoset_fft (SURVEY.md §3.2) ----
    uint4 *d_in = ctx->g_c.as<uint4>(), *d_aux = d_in + batch * n_in * 2;
    ZK_CUDA(cudaMemcpyAsync(d_in, inputs, batch * n_in * 32, cudaMemcpyHostToDevice, st));
    ZK_CUDA(cudaMemcpyAsync(d_aux, aux, batch * n_aux * 32, cudaMemcpyHostToDevice, st));
    // B-query scalars (inputs|B ++ aux|B ++ [1, s]) depend only on the assignment: build them first and start the G2 MSM
    // on the second lane, so its latency-bound tail overlaps the NTTs and the G1 MSMs of this lane.
    uint4 *scal2 = ctx->g_scal2.as<uint4>();
    if (bi_idx.size()) k_gather32<<<dim3((unsigned)((bi_idx.size() + 255) / 256), (unsigned)batch), 256, 0, st>>>(d_in, n_in, d_biidx, bi_idx.size(), scal2, nB, 0);
    if (ba_idx.size()) k_gather32<<<dim3((unsigned)((ba_idx.size() + 255) / 256), (unsigned)batch), 256, 0, st>>>(d_aux, n_aux, d_baidx, ba_idx.size(), scal2, nB, bi_idx.size());
    k_put_terms<<<(unsigned)((batch + 63) / 64), 64, 0, st>>>((const uint4 *)d_terms, 0, 2, 2, scal2, nB, nB - 2, batch);
    LaneEvents ev;
    ev.lane2 = lane2; ev.lane3 = lane3; ev.lane4 = lane4;
    ZK_TRY(ev.create());
    cudaEvent_t ev_b = ev.b, ev_g2 = ev.g2, ev_a = ev.a, ev_l3 = ev.l3, ev_l4 = ev.l4;
    ZK_CUDA(cudaEventRecord(ev_b, st));
    ZK_CUDA(cudaStreamWaitEvent(lane2->stream, ev_b, 0));
    ev.lanes_started = true;
    ZK_TRY(zk_msm_run(lane2, p->b2, scal2, nB, batch));
    ZK_CUDA(cudaMemcpyAsync(d_gb, lane2->result.p, batch * sizeof(G2XYZZ), cudaMemcpyDeviceToDevice, lane2->stream));
    ZK_CUDA(cudaEventRecord(ev_g2, lane2->stream));
    // third / fourth lane: g_a = MSM(a', inputs ++ aux|A ++ [1, r]) and g_b1 = MSM(b_g1', B scalars) need only the assignment too: their
    // scalars are built and the events recorded here, the MSMs themselves are enqueued after the longer chains (below)
    uint4 *scal3 = ctx->g_scal3.as<uint4>();
    ZK_CUDA(cudaMemcpy2DAsync(scal3, nA * 32, d_in, n_in * 32, n_in * 32, batch, cudaMemcpyDeviceToDevice, st));
    if (a_idx.size()) k_gather32<<<dim3((unsigned)((a_idx.size() + 255) / 256), (unsigned)batch), 256, 0, st>>>(d_aux, n_aux, d_aidx, a_idx.size(), scal3, nA, n_in);
    k_put_terms<<<(unsigned)((batch + 63) / 64), 64, 0, st>>>((const uint4 *)d_terms, 0, 1, 2, scal3, nA, nA - 2, batch);
    ZK_CUDA(cudaEventRecord(ev_a, st));
    ZK_CUDA(cudaStreamWaitEvent(lane3->stream, ev_a, 0));
    ZK_CUDA(cudaStreamWaitEvent(lane4->stream, ev_b, 0));              // the B scalars (scal2) are complete at ev_b
    if (r1cs) {
        ZK_TRY(ctx->g_b.reserve(batch * (n_in + n_aux) * 32));       // z in Montgomery form
        ZK_TRY(zk_fr_witness_to_mont(ctx, d_in, n_in, d_aux, n_aux, batch, ctx->g_b.p));
        for (int w = 0; w < 3; w++)
            ZK_TRY(zk_fr_r1cs_eval(ctx, r1cs->d_row_ptr[w], r1cs->d_col[w], r1cs->d_coeff[w], ctx->g_b.p, r1cs->n_c, n_in, n_in + n_aux, log_m, w, batch, ctx->g_a.p));
    } else {
        const uint64_t *evs[3] = {a_ev, b_ev, c_ev};
        for (int w = 0; w < 3; w++) {
            ZK_CUDA(cudaMemcpyAsync(ctx->g_b.p, evs[w], batch * n_c * 32, cudaMemcpyHostToDevice, st));
            ZK_TRY(zk_fr_load_evals(ctx, ctx->g_b.p, n_c, log_m, w, batch, ctx->g_a.p));
        }
    }
    ZK_TRY(zk_ntt_run(ctx, ctx->g_a.p, log_m, ZK_NTT_IFFT, 3 * batch));
    ZK_TRY(zk_ntt_run(ctx, ctx->g_a.p, log_m, ZK_NTT_COSET_FFT, 3 * batch));
    ZK_TRY(zk_fr_quotient(ctx, ctx->g_a.p, log_m, batch, ctx->g_h.p));
    ZK_TRY(zk_ntt_run(ctx, ctx->g_h.p, log_m, ZK_NTT_ICOSET_FFT, batch));
    // ---- H' = sum h_i * h[i] - rs * delta ----
    uint4 *scal = ctx->g_scal.as<uint4>();
    ZK_TRY(zk_fr_into_repr(ctx, ctx->g_h.p, log_m, m - 1, nH, batch, scal));
    k_put_terms<<<(unsigned)((batch + 63) / 64), 64, 0, st>>>((const uint4 *)d_terms, 3, 3, 1, scal, nH, m - 1, batch);
    ZK_TRY(zk_msm_run(ctx, p->h, scal, nH, batch));
    ZK_CUDA(cudaMemcpyAsync(d_H, ctx->result.p, batch * sizeof(G1XYZZ), cudaMemcpyDeviceToDevice, st));
    // (the host enqueues the LONGEST chains first — G2 above, NTTs -> H here — and only then the two shorter lanes below: with ~130 launches
    //  per proof the order in which they reach the streams is worth ~0.3 ms of single-proof latency)
    // lane 3: g_a, then s * g_a; lane 4: g_b1, then r * g_b1 — each variable-base multiplication needs only its own lane's MSM, and
    // both run under the NTT -> H -> L chain of the first lane
    ZK_TRY(zk_msm_run(lane3, p->a, scal3, nA, batch));
    ZK_CUDA(cudaMemcpyAsync(d_ga, lane3->result.p, batch * sizeof(G1XYZZ), cudaMemcpyDeviceToDevice, lane3->stream));
    const int glv = p->subgroup_checked ? 1 : 0;
    k_scale_points<<<(unsigned)batch, SCALE_T, 0, lane3->stream>>>(d_ga, d_gb1, (const uint32_t *)d_terms, batch, 0, glv, d_T);
    ZK_CUDA(cudaEventRecord(ev_l3, lane3->stream));
    ZK_TRY(zk_msm_run(lane4, p->b1, scal2, nB, batch));
    ZK_CUDA(cudaMemcpyAsync(d_gb1, lane4->result.p, batch * sizeof(G1XYZZ), cudaMemcpyDeviceToDevice, lane4->stream));
    k_scale_points<<<(unsigned)batch, SCALE_T, 0, lane4->stream>>>(d_ga, d_gb1, (const uint32_t *)d_terms, batch, 1, glv, d_T);
    ZK_CUDA(cudaEventRecord(ev_l4, lane4->stream));
    // ---- assignments (already on the device: d_in, d_aux) ----
    // L
    ZK_TRY(zk_msm_run(ctx, p->l, d_aux, n_aux, batch));
    ZK_CUDA(cudaMemcpyAsync(d_L, ctx->result.p, batch * sizeof(G1XYZZ), cudaMemcpyDeviceToDevice, st));
    ZK_CUDA(cudaStreamWaitEvent(st, ev_l3, 0));                       // join: g_a and s * g_a from the third lane
    ZK_CUDA(cudaStreamWaitEvent(st, ev_l4, 0));                       // join: r * g_b1 from the fourth
    ZK_CUDA(cudaStreamWaitEvent(st, ev_g2, 0));                       // join: g_b (G2) is ready in d_gb
    // ---- assembly + Proof::write ----
    k_finish_proofs<<<(unsigned)((batch + 31) / 32), 96, 0, st>>>(d_ga, d_gb, d_T, d_H, d_L, batch, d_proofs);
    ZK_CUDA(cudaGetLastError());
    ZK_CUDA(cudaMemcpyAsync(proofs_out, d_proofs, batch * 192, cudaMemcpyDeviceToHost, st));
    int rc = zk_check_err_flag(ctx);    // synchronises this lane (which has joined the second); reports non-canonical scalars
    std::string msg = rc ? zk_last_error() : "";
    int rcb = zk_check_err_flag(lane2), rcc = zk_check_err_flag(lane3), rcd = zk_check_err_flag(lane4);
    if (rc) zk_set_error("%s", msg.c_str());
    ev.completed = true;                // every lane has been synchronised and its error flag read
    return rc ? rc : (rcb ? rcb : (rcc ? rcc : rcd));
}

extern "C" int zk_groth16_prove_batch(zk_ctx *ctx, const zk_params *p, size_t batch,
                                      const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t n_c,
                                      const uint64_t *inputs, size_t n_in, const uint64_t *aux, size_t n_aux,
                                      const uint8_t *d1, const uint8_t *d2, const uint8_t *d3,
                                      const uint64_t *r, const uint64_t *s, uint8_t *out) {
    if (!a || !b || !c || !inputs || !aux || !r || !s || !out) { zk_set_error("zk_groth16_prove_batch: NULL argument"); return ZK_ERR_INVALID; }
    if (batch == 0) { zk_set_error("zk_groth16_prove_batch: empty batch"); return ZK_ERR_INVALID; }
    for (size_t o = 0; o < batch; o += PROVE_CHUNK) {
        size_t k = batch - o < PROVE_CHUNK ? batch - o : PROVE_CHUNK;
        ZK_TRY(prove_impl(ctx, p, k, a + o * n_c * 4, b + o * n_c * 4, c + o * n_c * 4, n_c, inputs + o * n_in * 4, n_in, aux + o * n_aux * 4, n_aux,
                          d1, d2, d3, r + o * 4, s + o * 4, out + o * 192));
    }
    return ZK_OK;
}
extern "C" int zk_groth16_prove(zk_ctx *ctx, const zk_params *p,
                                const uint64_t *a, const uint64_t *b, const uint64_t *c, size_t n_c,
                                const uint64_t *inputs, size_t n_in, const uint64_t *aux, size_t n_aux,
                                const uint8_t *d1, const uint8_t *d2, const uint8_t *d3,
                                const uint64_t r[4], const uint64_t s[4], uint8_t out[192]) {
    return prove_impl(ctx, p, 1, a, b, c, n_c, inputs, n_in, aux, n_aux, d1, d2, d3, r, s, out);
}

// ---- fixed constraint system on the device (SURVEY.md §8 f4) ---------------------------------------------------------
extern "C" void zk_r1cs_free(zk_r1cs *q) {
    if (!q) return;
    cudaSetDevice(q->device);
    for (int w = 0; w < 3; w++) { if (q->d_row_ptr[w]) cudaFree(q->d_row_ptr[w]); if (q->d_col[w]) cudaFree(q->d_col[w]); if (q->d_coeff[w]) cudaFree(q->d_coeff[w]); }
    delete q;
}
extern "C" int zk_r1cs_load(zk_ctx *ctx, size_t n_constraints, size_t n_inputs, size_t n_aux,
                            const uint32_t *a_row_ptr, const uint32_t *a_col, const uint64_t *a_coeff,
                            const uint32_t *b_row_ptr, const uint32_t *b_col, const uint64_t *b_coeff,
                            const uint32_t *c_row_ptr, const uint32_t *c_col, const uint64_t *c_coeff, zk_r1cs **out) {
    if (!ctx || !out || !a_row_ptr || !b_row_ptr || !c_row_ptr) { zk_set_error("zk_r1cs_load: NULL argument"); return ZK_ERR_INVALID; }
    if (n_constraints == 0 || n_inputs == 0) { zk_set_error("zk_r1cs_load: empty constraint system"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    const uint32_t *rp[3] = {a_row_ptr, b_row_ptr, c_row_ptr}, *cl[3] = {a_col, b_col, c_col};
    const uint64_t *cf[3] = {a_coeff, b_coeff, c_coeff};
    const size_t nv = n_inputs + n_aux;
    zk_r1cs *q = new zk_r1cs();
    q->device = ctx->device; q->n_c = n_constraints; q->n_in = n_inputs; q->n_aux = n_aux;
    q->a_aux_density.assign(n_aux ? n_aux : 1, 0); q->b_input_density.assign(n_inputs, 0); q->b_aux_density.assign(n_aux ? n_aux : 1, 0);
    for (int w = 0; w < 3; w++) {
        size_t nnz = rp[w][n_constraints];
        q->nnz[w] = nnz;
        if (rp[w][0] != 0 || (nnz && (!cl[w] || !cf[w]))) { zk_r1cs_free(q); zk_set_error("zk_r1cs_load: malformed CSR"); return ZK_ERR_INVALID; }
        for (size_t j = 0; j < n_constraints; j++) if (rp[w][j] > rp[w][j + 1]) { zk_r1cs_free(q); zk_set_error("zk_r1cs_load: row_ptr not monotone"); return ZK_ERR_INVALID; }
        for (size_t k = 0; k < nnz; k++) {
            uint32_t v = cl[w][k];
            if (v >= nv) { zk_r1cs_free(q); zk_set_error("zk_r1cs_load: variable index %u out of range", v); return ZK_ERR_INVALID; }
            if (w == 0 && v >= n_inputs) q->a_aux_density[v - n_inputs] = 1;
            if (w == 1) { if (v >= n_inputs) q->b_aux_density[v - n_inputs] = 1; else q->b_input_density[v] = 1; }
        }
        cudaError_t e1 = cudaMalloc(&q->d_row_ptr[w], (n_constraints + 1) * 4), e2 = cudaMalloc(&q->d_col[w], (nnz + 1) * 4), e3 = cudaMalloc(&q->d_coeff[w], (nnz + 1) * 32);
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) { zk_r1cs_free(q); zk_set_error("zk_r1cs_load: cudaMalloc failed"); return ZK_ERR_CUDA; }
        ZK_CUDA(cudaMemcpyAsync(q->d_row_ptr[w], rp[w], (n_constraints + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (nnz) {
            ZK_CUDA(cudaMemcpyAsync(q->d_col[w], cl[w], nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
            ZK_TRY(ctx->stage_a.reserve(nnz * 32));
            ZK_CUDA(cudaMemcpyAsync(ctx->stage_a.p, cf[w], nnz * 32, cudaMemcpyHostToDevice, ctx->stream));
            ZK_TRY(zk_fr_to_mont(ctx, ctx->stage_a.p, nnz, q->d_coeff[w]));
            ZK_CUDA(cudaStreamSynchronize(ctx->stream));
        }
    }
    int r = zk_check_err_flag(ctx);
    if (r) { zk_r1cs_free(q); return r; }
    *out = q;
    return ZK_OK;
}
extern "C" int zk_groth16_prove_witness_batch(zk_ctx *ctx, const zk_params *p, const zk_r1cs *q, size_t batch,
                                              const uint64_t *inputs, const uint64_t *aux, const uint64_t *r, const uint64_t *s, uint8_t *proofs_out) {
    if (!q) { zk_set_error("zk_groth16_prove_witness_batch: NULL constraint system"); return ZK_ERR_INVALID; }
    if (q->device != ctx->device) { zk_set_error("constraint system lives on device %d, context on %d", q->device, ctx->device); return ZK_ERR_INVALID; }
    if (!inputs || !aux || !r || !s || !proofs_out || batch == 0) { zk_set_error("zk_groth16_prove_witness_batch: bad argument"); return ZK_ERR_INVALID; }
    for (size_t o = 0; o < batch; o += PROVE_CHUNK) {
        size_t k = batch - o < PROVE_CHUNK ? batch - o : PROVE_CHUNK;
        ZK_TRY(prove_impl(ctx, p, k, nullptr, nullptr, nullptr, 0, inputs + o * q->n_in * 4, q->n_in, aux + o * q->n_aux * 4, q->n_aux, nullptr, nullptr, nullptr,
                          r + o * 4, s + o * 4, proofs_out + o * 192, q));
    }
    return ZK_OK;
}

// ---- generate_parameters (bellman groth16 generator.rs; reference calls core/proofs/src/setup.rs:28,59) ---------------------------
// Same algebra as bellman, on the device: powers of tau -> IFFT = the Lagrange coefficients at tau; at / bt / ct per variable = the
// coefficients summed over each matrix column (zk_setup_qap); the query scalars in CrsLayout order; one fixed-base launch for all G1
// scalars and one for all G2 scalars (zk_fixed_base); then the window tables as for a loaded CRS.  Every group element is unique and
// so is its uncompressed encoding: zk_params_write of the result equals what Parameters::write emits for the same inputs.
namespace {
const uint64_t FR_R[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
bool fr_canonical(const uint64_t *k) {
    for (int i = 3; i >= 0; i--) if (k[i] != FR_R[i]) return k[i] < FR_R[i];
    return false;
}
bool fr_zero(const uint64_t *k) { return !(k[0] | k[1] | k[2] | k[3]); }
// the trapdoor and everything derived from it (powers of tau, Lagrange coefficients, at / bt / ct, the query scalars) is the
// setup's toxic waste: the staging buffers that held it are cleared however the call ends
struct ClearTrapdoor {
    zk_ctx *ctx;
    ~ClearTrapdoor() {
        for (DevBuf *b : {&ctx->g_a, &ctx->g_b, &ctx->g_c, &ctx->g_h, &ctx->g_scal, &ctx->g_scal2, &ctx->ntt_tmp})
            if (b->p) cudaMemsetAsync(b->p, 0, b->cap, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    }
};
}  // namespace

extern "C" int zk_groth16_generate(zk_ctx *ctx, const zk_r1cs *q, const uint8_t g1[96], const uint8_t g2[192], const uint64_t alpha[4],
                                   const uint64_t beta[4], const uint64_t gamma[4], const uint64_t delta[4], const uint64_t tau[4], zk_params **out) {
    if (!ctx || !q || !g1 || !g2 || !alpha || !beta || !gamma || !delta || !tau || !out) { zk_set_error("zk_groth16_generate: NULL argument"); return ZK_ERR_INVALID; }
    if (q->device != ctx->device) { zk_set_error("constraint system lives on device %d, context on %d", q->device, ctx->device); return ZK_ERR_INVALID; }
    const uint64_t *sc[5] = {tau, alpha, beta, gamma, delta};
    static const char *names[5] = {"tau", "alpha", "beta", "gamma", "delta"};
    for (int k = 0; k < 5; k++) if (!fr_canonical(sc[k])) { zk_set_error("%s is not canonical (>= r)", names[k]); return ZK_ERR_NOT_CANONICAL; }
    // gamma, delta: bellman's own UnexpectedIdentity; alpha, beta: zk_params_load would reject the vk points; tau: the h query would
    // hold the identity, which Parameters::read rejects
    for (int k : {3, 4, 1, 2, 0}) if (fr_zero(sc[k])) { zk_set_error("UnexpectedIdentity: %s = 0", names[k]); return ZK_ERR_UNEXPECTED_IDENTITY; }
    ZK_TRY(zk_use_device(ctx));
    const size_t n_c = q->n_c, n_in = q->n_in, n_aux = q->n_aux, nv = n_in + n_aux;
    unsigned log_m = 0;
    size_t m = 1;
    while (m < n_c + n_in) { m <<= 1; log_m++; }
    if (log_m > 28 || m - 1 >= CRS_POINT_LIMIT || nv >= CRS_POINT_LIMIT) {
        zk_set_error("PolynomialDegreeTooLarge: domain 2^%u, %zu variables (limits 2^28, %u points per vector)", log_m, nv, CRS_POINT_LIMIT);
        return ZK_ERR_POLY_DEGREE_TOO_LARGE;
    }
    ClearTrapdoor clear{ctx};
    cudaStream_t st = ctx->stream;
    // ---- staging (reserved up front: a buffer that grows later would be freed without being cleared) ----
    const size_t nnz_max = q->nnz[0] > q->nnz[1] ? (q->nnz[0] > q->nnz[2] ? q->nnz[0] : q->nnz[2]) : (q->nnz[1] > q->nnz[2] ? q->nnz[1] : q->nnz[2]);
    const size_t g1_cap = m + n_aux + 2 * (nv + 2) + 3 + n_in + 8;
    ZK_TRY(ctx->g_a.reserve(m * 32));                        // powers of tau, then the Lagrange coefficients
    ZK_TRY(ctx->ntt_tmp.reserve(m * 32));
    ZK_TRY(ctx->g_h.reserve((3 * nv + 16) * 32));            // at | bt | ct, the constants, the five scalars
    ZK_TRY(ctx->g_b.reserve((nnz_max + nv + 1) * 32));       // column-sorted entries and task sums (ping-pong)
    ZK_TRY(ctx->g_c.reserve((nnz_max + nv + 1) * 32));
    ZK_TRY(ctx->g_scal.reserve(g1_cap * 32));                // G1 scalars in CrsLayout order
    ZK_TRY(ctx->g_scal2.reserve((nv + 8) * 32));             // G2 scalars
    auto rnd = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t scratch_words = 3 * (nv + 1) + 2 * (nv / 2048 + 8) + 64;
    ZK_TRY(ctx->g_misc.reserve(rnd(288) + rnd(sizeof(G1Affine)) + rnd(sizeof(G2Affine)) + rnd(16) + 3 * rnd((nv + 1) * 4) + rnd(scratch_words * 4)));
    uint8_t *mp = ctx->g_misc.as<uint8_t>();
    auto carve = [&](size_t bytes) { uint8_t *r = mp; mp += rnd(bytes); return r; };
    uint8_t *d_enc = carve(288);
    G1Affine *d_gen1 = (G1Affine *)carve(sizeof(G1Affine));
    G2Affine *d_gen2 = (G2Affine *)carve(sizeof(G2Affine));
    int *d_flag = (int *)carve(16);
    uint32_t *pos_a = (uint32_t *)carve((nv + 1) * 4), *pos_b = (uint32_t *)carve((nv + 1) * 4), *scratch = (uint32_t *)carve(scratch_words * 4);
    uint4 *abc = ctx->g_h.as<uint4>(), *consts = abc + 2 * 3 * nv, *d_in = consts + 2 * 8;
    uint4 *P = ctx->g_a.as<uint4>(), *scal1 = ctx->g_scal.as<uint4>(), *scal2 = ctx->g_scal2.as<uint4>();
    // ---- generators: checked decoding (on the curve, in the r-torsion, not the identity) ----
    ZK_CUDA(cudaMemcpyAsync(d_enc, g1, 96, cudaMemcpyHostToDevice, st));
    ZK_CUDA(cudaMemcpyAsync(d_enc + 96, g2, 192, cudaMemcpyHostToDevice, st));
    zkcodec::k_decode_uncompressed<Fq><<<1, 128, 0, st>>>(d_enc, 1, 1, 1, d_gen1, ctx->d_err + 1);
    zkcodec::k_decode_uncompressed<Fq2><<<1, 128, 0, st>>>(d_enc + 96, 1, 1, 1, d_gen2, ctx->d_err + 1);
    ZK_CUDA(cudaGetLastError());
    ZK_TRY(zk_check_err_flag(ctx));
    // ---- powers of tau, h, Lagrange coefficients ----
    for (int k = 0; k < 5; k++) ZK_CUDA(cudaMemcpyAsync(d_in + 2 * k, sc[k], 32, cudaMemcpyHostToDevice, st));
    ZK_CUDA(cudaMemsetAsync(d_flag, 0, 16, st));
    ZK_TRY(zk_setup_powers(ctx, d_in, log_m, consts, d_flag, P, scal1));        // h = G1 scalars [0, m - 1) (CrsLayout: o_h = 0)
    int flags[2] = {0, 0};
    ZK_CUDA(cudaMemcpyAsync(flags, d_flag, 4, cudaMemcpyDeviceToHost, st));
    ZK_CUDA(cudaStreamSynchronize(st));
    if (flags[0]) { zk_set_error("UnexpectedIdentity: tau^m = 1 (m = 2^%u), the h query would contain the identity", log_m); return ZK_ERR_UNEXPECTED_IDENTITY; }
    ZK_TRY(zk_ntt_run(ctx, P, log_m, ZK_NTT_IFFT, 1));
    // ---- at, bt, ct (the `input_i * 0 = 0` rows add L_{n_c + i} to at) ----
    for (int w = 0; w < 3; w++)
        ZK_TRY(zk_setup_qap(ctx, q->d_row_ptr[w], q->d_col[w], q->d_coeff[w], n_c, q->nnz[w], nv, P, w == 0 ? n_in : 0, scratch,
                            ctx->g_b.p, ctx->g_c.p, abc + 2 * w * nv));
    // ---- query sizes: identities dropped from a, b_g1, b_g2 by value; an l scalar of zero is an unconstrained variable ----
    ZK_TRY(zk_setup_flags(ctx, abc, consts, nv, n_in, pos_a, pos_b, d_flag + 1, scratch));
    uint32_t cnt_ab[2] = {0, 0};
    ZK_CUDA(cudaMemcpyAsync(cnt_ab, pos_a + nv, 4, cudaMemcpyDeviceToHost, st));
    ZK_CUDA(cudaMemcpyAsync(cnt_ab + 1, pos_b + nv, 4, cudaMemcpyDeviceToHost, st));
    ZK_CUDA(cudaMemcpyAsync(flags + 1, d_flag + 1, 4, cudaMemcpyDeviceToHost, st));
    ZK_CUDA(cudaStreamSynchronize(st));
    if (flags[1]) { zk_set_error("UnconstrainedVariable: an aux variable's l query point is the identity"); return ZK_ERR_UNCONSTRAINED_VARIABLE; }
    const size_t cnt[6] = {n_in, m - 1, n_aux, cnt_ab[0], cnt_ab[1], cnt_ab[1]};
    CrsLayout L(cnt);
    // ---- the scalars in CrsLayout order: h' | l | a' | b_g1' | vk1 and b_g2' | vk2 ----
    auto put = [&](uint4 *dst, int k) { return cudaMemcpyAsync(dst, d_in + 2 * k, 32, cudaMemcpyDeviceToDevice, st); };
    enum { TAU, ALPHA, BETA, GAMMA, DELTA };
    ZK_CUDA(put(scal1 + 2 * (L.o_h + m - 1), DELTA));
    ZK_CUDA(put(scal1 + 2 * (L.o_a + cnt[3]), ALPHA)); ZK_CUDA(put(scal1 + 2 * (L.o_a + cnt[3] + 1), DELTA));
    ZK_CUDA(put(scal1 + 2 * (L.o_b1 + cnt[4]), BETA)); ZK_CUDA(put(scal1 + 2 * (L.o_b1 + cnt[4] + 1), DELTA));
    ZK_CUDA(put(scal1 + 2 * L.o_vk1, ALPHA)); ZK_CUDA(put(scal1 + 2 * (L.o_vk1 + 1), BETA)); ZK_CUDA(put(scal1 + 2 * (L.o_vk1 + 2), DELTA));
    ZK_CUDA(put(scal2 + 2 * cnt[5], BETA)); ZK_CUDA(put(scal2 + 2 * (cnt[5] + 1), DELTA));
    ZK_CUDA(put(scal2 + 2 * (L.n_b2), BETA)); ZK_CUDA(put(scal2 + 2 * (L.n_b2 + 1), GAMMA)); ZK_CUDA(put(scal2 + 2 * (L.n_b2 + 2), DELTA));
    ZK_TRY(zk_setup_fill(ctx, abc, consts, nv, n_in, pos_a, pos_b, scal1 + 2 * L.o_l, scal1 + 2 * (L.o_vk1 + 3), scal1 + 2 * L.o_a, scal1 + 2 * L.o_b1, scal2));
    // ---- the group elements: one fixed-base launch per group ----
    ZK_TRY(ctx->stage_b.reserve((L.g1_total + 8) * sizeof(G1Affine)));
    ZK_TRY(ctx->stage_c.reserve((L.g2_total + 8) * sizeof(G2Affine)));
    ZK_TRY(zk_fixed_base(ctx, 1, d_gen1, scal1, L.g1_total, ctx->stage_b.p));
    ZK_TRY(zk_fixed_base(ctx, 2, d_gen2, scal2, L.g2_total, ctx->stage_c.p));
    ZK_TRY(params_from_device(ctx, L, ctx->stage_b.as<G1Affine>(), ctx->stage_c.as<G2Affine>(), out));
    (*out)->subgroup_checked = true;     // every point is a multiple of a checked generator
    return ZK_OK;
}
