// Device work of Groth16 parameter generation (bellman 0.1.0 groth16::generate_parameters; reference call sites
// core/proofs/src/setup.rs:28,59 through generate_random_parameters) and the batched fixed-base multiplication it rests on,
// which zk_scalar_mul_many uses as well.  The orchestration is zk_groth16_generate in groth16.cu.
//
//   zk_fixed_base          k_fb_bases (2^(C w) g, one warp-cooperative doubling chain) -> k_fb_table (d 2^(C w) g, thread per
//                          entry) -> k_fixed_base (thread per scalar: one mixed addition per non-zero signed digit, affine output
//                          with one inversion per warp)
//   zk_setup_powers        tau^i (Montgomery, for the IFFT) and the h scalars tau^i t(tau) / delta (canonical)
//   zk_setup_qap           at / bt / ct = the Lagrange coefficients summed per column: counting sort of the CSR entries by column
//                          (histogram, scan, scatter), then bounded segmented sums (setup.cuh)
//   zk_setup_flags/_fill   the non-zero filters of the a / b queries (scan positions) and the ic / l / a / b scalars
#define ZK_SEMI_HOT 1   // Fq product inlined into the (noinline) point operations, as in groth16.cu
#include <stdlib.h>
#include "internal.h"
#include "curve_coop.cuh"
#include "msm.cuh"             // zkmsm::exclusive_scan
#include "msm_warp_scan.cuh"   // zkmsm::ba_warp_products
#include "setup.cuh"

using namespace zksetup;

// Window bits of the fixed-base tables, chosen by measurement (tools/setup_bench.py on 2^20 G1 scalars, table build included:
// c = 6 / 8 / 10 / 12 -> 55.2 / 48.8 / 44.6 / 42.6 ms on a B200; DESIGN.md §3a).  Experiment builds (make EXPERIMENTS=1) read ZK_FB_C
// to repeat that sweep.
static constexpr int FB_C = 12;

namespace {
constexpr int FB_T = 128;

// affine conversion of one point per lane, one inversion per warp (all 32 lanes must call it)
template <class F>
__device__ __forceinline__ Affine<F> fb_warp_affine(const XYZZ<F> &q) {
    F others, all;
    zkmsm::ba_warp_products(fb_denominator(q), others, all);
    return fb_affine(q, all.inverse() * others);
}
// bases[w] = 2^(C w) g: warp 0 runs the doubling chain (three cooperative stages per doubling), then both warps convert
template <class F, int C>
__global__ void __launch_bounds__(64) k_fb_bases(const Affine<F> *__restrict__ g, Affine<F> *__restrict__ bases) {
    constexpr int W = FbGeom<C>::W;
    static_assert(W <= 64, "one block of 64 threads converts the window bases");
    __shared__ XYZZ<F> chain[W];
    if (threadIdx.x < 32) {
        XYZZ<F> p = XYZZ<F>::from_affine(*g);
        for (int w = 0; w < W; w++) {
            if (threadIdx.x == 0) chain[w] = p;
            if (w + 1 < W) for (int i = 0; i < C; i++) zkcoop::dbl(p);
        }
    }
    __syncthreads();
    const XYZZ<F> q = threadIdx.x < W ? chain[threadIdx.x] : XYZZ<F>::inf();
    const Affine<F> a = fb_warp_affine(q);
    if (threadIdx.x < W) bases[threadIdx.x] = a;
}
// tbl[w][d - 1] = d bases[w], thread per entry (the entry count is a multiple of 32: every warp is full)
template <class F, int C>
__global__ void __launch_bounds__(FB_T) k_fb_table(const Affine<F> *__restrict__ bases, Affine<F> *__restrict__ tbl) {
    const uint32_t e = blockIdx.x * FB_T + threadIdx.x;
    const bool live = e < (uint32_t)FbGeom<C>::ENTRIES;
    const XYZZ<F> q = live ? fb_small_mul(bases[e / FbGeom<C>::HALF], e % FbGeom<C>::HALF + 1) : XYZZ<F>::inf();
    const Affine<F> a = fb_warp_affine(q);
    if (live) tbl[e] = a;
}
// out[i] = k_i g (affine), k_i any 256-bit value (8 LE u32 words)
template <class F, int C>
__global__ void __launch_bounds__(FB_T) k_fixed_base(const Affine<F> *__restrict__ tbl, const uint32_t *__restrict__ scalars, size_t n,
                                                     Affine<F> *__restrict__ out) {
    const size_t i = (size_t)blockIdx.x * FB_T + threadIdx.x;
    XYZZ<F> acc = XYZZ<F>::inf();
    if (i < n) {
        uint32_t k[8];
        const uint4 *s = reinterpret_cast<const uint4 *>(scalars + i * 8);
        const uint4 s0 = s[0], s1 = s[1];
        k[0] = s0.x; k[1] = s0.y; k[2] = s0.z; k[3] = s0.w; k[4] = s1.x; k[5] = s1.y; k[6] = s1.z; k[7] = s1.w;
        acc = fb_walk<F, C>(tbl, k);
    }
    const Affine<F> a = fb_warp_affine(acc);     // every lane takes part, live or not
    if (i < n) out[i] = a;
}

template <class F, int C>
int fixed_base_t(zk_ctx *ctx, const void *d_base, const void *d_scalars, size_t n, void *d_out) {
    cudaStream_t st = ctx->stream;
    constexpr int E = FbGeom<C>::ENTRIES;
    ZK_TRY(ctx->fb_tbl.reserve((size_t)(E + FbGeom<C>::W) * sizeof(Affine<F>)));
    Affine<F> *tbl = ctx->fb_tbl.as<Affine<F>>(), *bases = tbl + E;
    k_fb_bases<F, C><<<1, 64, 0, st>>>((const Affine<F> *)d_base, bases);
    k_fb_table<F, C><<<(E + FB_T - 1) / FB_T, FB_T, 0, st>>>(bases, tbl);
    for (size_t o = 0; o < n; o += (size_t)FB_T << 20) {        // grid.x stays far below its limit
        size_t k = n - o < ((size_t)FB_T << 20) ? n - o : ((size_t)FB_T << 20);
        k_fixed_base<F, C><<<(unsigned)((k + FB_T - 1) / FB_T), FB_T, 0, st>>>(tbl, (const uint32_t *)d_scalars + o * 8, k, (Affine<F> *)d_out + o);
    }
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}
template <class F>
int fixed_base_c(zk_ctx *ctx, const void *d_base, const void *d_scalars, size_t n, void *d_out) {
#ifdef ZK_EXPERIMENTS
    if (const char *e = getenv("ZK_FB_C")) {
        switch (atoi(e)) {
        case 6: return fixed_base_t<F, 6>(ctx, d_base, d_scalars, n, d_out);
        case 8: return fixed_base_t<F, 8>(ctx, d_base, d_scalars, n, d_out);
        case 10: return fixed_base_t<F, 10>(ctx, d_base, d_scalars, n, d_out);
        default: break;
        }
    }
#endif
    return fixed_base_t<F, FB_C>(ctx, d_base, d_scalars, n, d_out);
}
}  // namespace

int zk_fixed_base(zk_ctx *ctx, int group, const void *d_base, const void *d_scalars, size_t n, void *d_out) {
    if (n == 0) return ZK_OK;
    return group == 1 ? fixed_base_c<Fq>(ctx, d_base, d_scalars, n, d_out) : fixed_base_c<Fq2>(ctx, d_base, d_scalars, n, d_out);
}

// ---- powers of tau, h scalars ----------------------------------------------------------------------------------------------
namespace {
// in: tau, alpha, beta, gamma, delta canonical.  consts (Montgomery): tau, alpha, beta, 1/gamma, 1/delta, t(tau)/delta.
// *flag = 1 when t(tau) = tau^m - 1 = 0 (tau an m-th root of unity: the h query would hold the identity).
__global__ void k_setup_consts(const Fr *__restrict__ in, unsigned log_m, Fr *__restrict__ consts, int *__restrict__ flag) {
    const Fr tau = Fr::from_canonical(in[0]);
    Fr tm = tau;
    for (unsigned i = 0; i < log_m; i++) tm = tm.sqr();
    const Fr zt = tm - Fr::one(), dinv = Fr::from_canonical(in[4]).inverse();
    consts[0] = tau; consts[1] = Fr::from_canonical(in[1]); consts[2] = Fr::from_canonical(in[2]);
    consts[3] = Fr::from_canonical(in[3]).inverse(); consts[4] = dinv; consts[5] = zt * dinv;
    *flag = zt.is_zero() ? 1 : 0;
}
constexpr uint32_t POW_CHUNK = 32;
// P[i] = tau^i for i < m (each thread raises tau to its chunk start, then multiplies along); h[i] = into_repr(tau^i t(tau)/delta), i < m - 1
__global__ void k_tau_powers(const Fr *__restrict__ consts, size_t m, Fr *__restrict__ P, Fr *__restrict__ h) {
    const size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * POW_CHUNK;
    if (i0 >= m) return;
    const Fr tau = consts[0], ztd = consts[5];
    const uint32_t e = (uint32_t)i0;            // m <= 2^28
    Fr p = tau.pow(&e, 1);
    for (size_t i = i0; i < i0 + POW_CHUNK && i < m; i++) {
        P[i] = p;
        if (i + 1 < m) h[i] = (p * ztd).to_canonical();
        p = p * tau;
    }
}
}  // namespace

int zk_setup_powers(zk_ctx *ctx, const void *d_in, unsigned log_m, void *d_consts, int *d_flag, void *d_P, void *d_h) {
    const size_t m = (size_t)1 << log_m;
    k_setup_consts<<<1, 1, 0, ctx->stream>>>((const Fr *)d_in, log_m, (Fr *)d_consts, d_flag);
    const size_t threads = (m + POW_CHUNK - 1) / POW_CHUNK;
    k_tau_powers<<<(unsigned)((threads + 127) / 128), 128, 0, ctx->stream>>>((const Fr *)d_consts, m, (Fr *)d_P, (Fr *)d_h);
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}

// ---- QAP evaluation at tau ----------------------------------------------------------------------------------------------
namespace {
__global__ void k_col_hist(const uint32_t *__restrict__ col, size_t nnz, uint32_t *__restrict__ hist) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nnz) atomicAdd(hist + col[k], 1u);
}
// entry k of row j lands at its column's next free slot with the value coeff_k L_j (the order inside a column is arbitrary:
// the sums are exact)
__global__ void k_col_scatter(const uint32_t *__restrict__ row_ptr, const uint32_t *__restrict__ col, const Fr *__restrict__ coeff,
                              const Fr *__restrict__ L, size_t n_c, uint32_t *__restrict__ cursor, Fr *__restrict__ vals) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_c) return;
    const Fr l = L[j];
    for (uint32_t k = row_ptr[j]; k < row_ptr[j + 1]; k++) vals[atomicAdd(cursor + col[k], 1u)] = coeff[k] * l;
}
__global__ void k_qap_count(const uint32_t *__restrict__ seg_off, size_t n_seg, uint32_t *__restrict__ cnt) {
    size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_seg) cnt[v] = qap_tasks_of(seg_off, v);
}
__global__ void k_qap_tasks(const uint32_t *__restrict__ seg_off, const uint32_t *__restrict__ task_off, size_t n_seg, const Fr *__restrict__ vals,
                            size_t max_tasks, Fr *__restrict__ out) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= max_tasks || t >= task_off[n_seg]) return;
    out[t] = qap_task_sum(seg_off, task_off, n_seg, vals, (uint32_t)t);
}
// out[v] = the column sum, plus L_{n_c + v} for the `input_v * 0 = 0` row of each input (A only)
__global__ void k_qap_final(const uint32_t *__restrict__ seg_off, const Fr *__restrict__ vals, size_t nv, const Fr *__restrict__ L_inputs,
                            size_t n_in, Fr *__restrict__ out) {
    size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    Fr s = qap_segment_value(seg_off, vals, v);
    if (L_inputs && v < n_in) s = s + L_inputs[v];
    out[v] = s;
}
}  // namespace

// scratch: u32 words, >= 3 (nv + 1) + 2 (nv / SCAN_B + 8) + 64; vals0 / vals1: max(nnz, nnz / QAP_T + nv) + 1 Fr each
int zk_setup_qap(zk_ctx *ctx, const uint32_t *d_row_ptr, const uint32_t *d_col, const void *d_coeff, size_t n_c, size_t nnz, size_t nv,
                 const void *d_L, size_t n_in_rows, uint32_t *scratch, void *d_vals0, void *d_vals1, void *d_out) {
    cudaStream_t st = ctx->stream;
    uint32_t *off0 = scratch, *off1 = off0 + nv + 1, *cnt = off1 + nv + 1, *scan_tmp = cnt + nv + 1;
    Fr *va = (Fr *)d_vals0, *vb = (Fr *)d_vals1;
    const Fr *L = (const Fr *)d_L;
    const unsigned gv = (unsigned)((nv + 255) / 256);
    ZK_CUDA(cudaMemsetAsync(cnt, 0, (nv + 1) * 4, st));
    if (nnz) k_col_hist<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(d_col, nnz, cnt);
    zkmsm::exclusive_scan<false>(cnt, off0, nv, scan_tmp, st);                  // column offsets
    ZK_CUDA(cudaMemcpyAsync(off1, off0, (nv + 1) * 4, cudaMemcpyDeviceToDevice, st));
    if (n_c) k_col_scatter<<<(unsigned)((n_c + 127) / 128), 128, 0, st>>>(d_row_ptr, d_col, (const Fr *)d_coeff, L, n_c, off1, va);
    size_t span = nnz, entries = nnz;           // bounds: longest segment, values in the current pass
    while (span > 1) {
        k_qap_count<<<gv, 256, 0, st>>>(off0, nv, cnt);
        zkmsm::exclusive_scan<false>(cnt, off1, nv, scan_tmp, st);
        size_t tasks = entries / QAP_T + nv;
        if (tasks > entries) tasks = entries;
        k_qap_tasks<<<(unsigned)((tasks + 127) / 128), 128, 0, st>>>(off0, off1, nv, va, tasks, vb);
        uint32_t *to = off0; off0 = off1; off1 = to;
        Fr *tv = va; va = vb; vb = tv;
        span = (span + QAP_T - 1) / QAP_T;
        entries = tasks;
    }
    k_qap_final<<<gv, 256, 0, st>>>(off0, va, nv, n_in_rows ? L + n_c : nullptr, n_in_rows, (Fr *)d_out);
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}

// ---- the query scalars ------------------------------------------------------------------------------------------------------
namespace {
// nz_a[v] = at_v != 0, nz_b[v] = bt_v != 0 (bellman drops identities from a, b_g1, b_g2 by value); *flag = 1 when an aux
// variable's l scalar beta at + alpha bt + ct is zero (SynthesisError::UnconstrainedVariable)
__global__ void k_setup_flags(const Fr *__restrict__ abc, const Fr *__restrict__ consts, size_t nv, size_t n_in, uint32_t *__restrict__ nz_a,
                              uint32_t *__restrict__ nz_b, int *__restrict__ flag) {
    size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    const Fr at = abc[v], bt = abc[nv + v], ct = abc[2 * nv + v];
    nz_a[v] = at.is_zero() ? 0 : 1;
    nz_b[v] = bt.is_zero() ? 0 : 1;
    if (v >= n_in && (consts[2] * at + consts[1] * bt + ct).is_zero()) atomicExch(flag, 1);
}
// G1 scalars in CrsLayout order: l[i] = (beta at + alpha bt + ct) / delta (aux), ic[i] = the same / gamma (inputs, after the three
// vk scalars), a and b_g1 compacted by the scan positions; G2: b_g2 = the same bt as b_g1
__global__ void k_setup_fill(const Fr *__restrict__ abc, const Fr *__restrict__ consts, size_t nv, size_t n_in, const uint32_t *__restrict__ pos_a,
                             const uint32_t *__restrict__ pos_b, Fr *__restrict__ l, Fr *__restrict__ ic, Fr *__restrict__ a, Fr *__restrict__ b1,
                             Fr *__restrict__ b2) {
    size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nv) return;
    const Fr at = abc[v], bt = abc[nv + v], ct = abc[2 * nv + v];
    const Fr comb = consts[2] * at + consts[1] * bt + ct;
    if (v < n_in) ic[v] = (comb * consts[3]).to_canonical();
    else l[v - n_in] = (comb * consts[4]).to_canonical();
    if (pos_a[v + 1] != pos_a[v]) a[pos_a[v]] = at.to_canonical();
    if (pos_b[v + 1] != pos_b[v]) { const Fr b = bt.to_canonical(); b1[pos_b[v]] = b; b2[pos_b[v]] = b; }
}
}  // namespace

// pos_a / pos_b: nv + 1 words each (exclusive scans; [nv] = the counts); scratch as for zk_setup_qap
int zk_setup_flags(zk_ctx *ctx, const void *d_abc, const void *d_consts, size_t nv, size_t n_in, uint32_t *pos_a, uint32_t *pos_b, int *d_flag,
                   uint32_t *scratch) {
    cudaStream_t st = ctx->stream;
    uint32_t *nz_a = scratch, *nz_b = nz_a + nv + 1, *scan_tmp = nz_b + nv + 1;
    k_setup_flags<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>((const Fr *)d_abc, (const Fr *)d_consts, nv, n_in, nz_a, nz_b, d_flag);
    zkmsm::exclusive_scan<false>(nz_a, pos_a, nv, scan_tmp, st);
    zkmsm::exclusive_scan<false>(nz_b, pos_b, nv, scan_tmp, st);
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}
int zk_setup_fill(zk_ctx *ctx, const void *d_abc, const void *d_consts, size_t nv, size_t n_in, const uint32_t *pos_a, const uint32_t *pos_b,
                  void *d_l, void *d_ic, void *d_a, void *d_b1, void *d_b2) {
    k_setup_fill<<<(unsigned)((nv + 255) / 256), 256, 0, ctx->stream>>>((const Fr *)d_abc, (const Fr *)d_consts, nv, n_in, pos_a, pos_b, (Fr *)d_l,
                                                                      (Fr *)d_ic, (Fr *)d_a, (Fr *)d_b1, (Fr *)d_b2);
    ZK_CUDA(cudaGetLastError());
    return ZK_OK;
}
