// CPU unit-test harness of parameter generation's per-thread device code (zero_chain_b200/csrc/setup.cuh), compiled with
// ZK_HOST_EMUL: signed-digit recoding, the fixed-base table walk, the affine conversion with a shared inverse, the bounded
// segmented column sums.  The passes of setup.cu are replayed here in plain loops.  Test infrastructure only.
#define ZK_HOST_EMUL 1
#include <string.h>
#include <vector>
#include "setup.cuh"
using namespace zksetup;

template <int C> static int t_recode(const uint32_t *k, int *digits) {
    uint32_t carry = 0;
    for (int w = 0; w < FbGeom<C>::W; w++) digits[w] = fb_digit<C>(k, w, carry);
    return (int)carry;        // must be 0: the last window absorbs the carry
}
// the table of setup.cu (k_fb_bases, k_fb_table): T[w][d - 1] = d 2^(C w) g
template <class F, int C> static std::vector<Affine<F>> t_table(const Affine<F> &g) {
    std::vector<Affine<F>> bases(FbGeom<C>::W), tbl(FbGeom<C>::ENTRIES);
    XYZZ<F> p = XYZZ<F>::from_affine(g);
    for (int w = 0; w < FbGeom<C>::W; w++) {
        bases[w] = p.to_affine();
        for (int i = 0; i < C; i++) p = p.dbl();
    }
    for (int e = 0; e < FbGeom<C>::ENTRIES; e++) tbl[e] = fb_small_mul(bases[e / FbGeom<C>::HALF], e % FbGeom<C>::HALF + 1).to_affine();
    return tbl;
}
template <class F, int C> static void t_walk(const uint32_t *g, const uint32_t *k, int n, uint32_t *out) {
    Affine<F> a; memcpy(&a, g, sizeof(a));
    std::vector<Affine<F>> tbl = t_table<F, C>(a);
    for (int i = 0; i < n; i++) { Affine<F> r = fb_walk<F, C>(tbl.data(), k + 8 * i).to_affine(); memcpy(out + i * sizeof(r) / 4, &r, sizeof(r)); }
}
// n affine inputs -> XYZZ with a non-trivial Z (2 P_i, kept as XYZZ), then the shared-inverse conversion of setup.cu's warps:
// lane i gets (product of all denominators)^-1 * (product of the others)
template <class F> static void t_normalize(const uint32_t *in, int n, uint32_t *out) {
    std::vector<XYZZ<F>> q(n);
    for (int i = 0; i < n; i++) { Affine<F> a; memcpy(&a, in + i * sizeof(a) / 4, sizeof(a)); q[i] = XYZZ<F>::from_affine(a).dbl(); }
    F all = F::one();
    for (int i = 0; i < n; i++) all = all * fb_denominator(q[i]);
    const F inv = all.inverse();
    for (int i = 0; i < n; i++) {
        F others = F::one();
        for (int j = 0; j < n; j++) if (j != i) others = others * fb_denominator(q[j]);
        Affine<F> r = fb_affine(q[i], inv * others);
        memcpy(out + i * sizeof(r) / 4, &r, sizeof(r));
    }
}
static std::vector<uint32_t> excl_scan(const std::vector<uint32_t> &c) {
    std::vector<uint32_t> o(c.size() + 1, 0);
    for (size_t i = 0; i < c.size(); i++) o[i + 1] = o[i] + c[i];
    return o;
}
extern "C" {
int emu_recode(const uint32_t *k, int c, int *digits) {
    switch (c) {
    case 6: return t_recode<6>(k, digits);
    case 8: return t_recode<8>(k, digits);
    case 10: return t_recode<10>(k, digits);
    case 12: return t_recode<12>(k, digits);
    default: return -1;
    }
}
int emu_windows(int c) { return c == 6 ? FbGeom<6>::W : c == 8 ? FbGeom<8>::W : c == 10 ? FbGeom<10>::W : FbGeom<12>::W; }
void emu_g1_walk(const uint32_t *g, const uint32_t *k, int n, int c, uint32_t *out) {
    if (c == 6) t_walk<Fq, 6>(g, k, n, out); else if (c == 8) t_walk<Fq, 8>(g, k, n, out); else if (c == 10) t_walk<Fq, 10>(g, k, n, out); else t_walk<Fq, 12>(g, k, n, out);
}
void emu_g2_walk(const uint32_t *g, const uint32_t *k, int n, int c, uint32_t *out) {
    if (c == 6) t_walk<Fq2, 6>(g, k, n, out); else if (c == 8) t_walk<Fq2, 8>(g, k, n, out); else t_walk<Fq2, 12>(g, k, n, out);
}
void emu_g1_normalize(const uint32_t *in, int n, uint32_t *out) { t_normalize<Fq>(in, n, out); }
void emu_g2_normalize(const uint32_t *in, int n, uint32_t *out) { t_normalize<Fq2>(in, n, out); }
// the column sums of one matrix: entries (col[k], val[k]) in any order (Montgomery Fr), nv columns -> out[nv]; returns the passes run
int emu_column_sums(const uint32_t *col, const uint32_t *vals_in, size_t nnz, size_t nv, uint32_t *out) {
    std::vector<uint32_t> hist(nv, 0);
    for (size_t k = 0; k < nnz; k++) hist[col[k]]++;
    std::vector<uint32_t> seg = excl_scan(hist), cur(seg.begin(), seg.end() - 1);
    std::vector<Fr> vals(nnz + 1);
    for (size_t k = 0; k < nnz; k++) memcpy(&vals[cur[col[k]]++], vals_in + 8 * k, 32);
    int passes = 0;
    for (size_t span = nnz; span > 1; span = (span + QAP_T - 1) / QAP_T, passes++) {
        std::vector<uint32_t> cnt(nv);
        for (size_t v = 0; v < nv; v++) cnt[v] = qap_tasks_of(seg.data(), v);
        std::vector<uint32_t> task = excl_scan(cnt);
        std::vector<Fr> next(task[nv] + 1);
        for (uint32_t t = 0; t < task[nv]; t++) next[t] = qap_task_sum(seg.data(), task.data(), nv, vals.data(), t);
        seg = task; vals = next;
    }
    for (size_t v = 0; v < nv; v++) { Fr s = qap_segment_value(seg.data(), vals.data(), v); memcpy(out + 8 * v, &s, 32); }
    return passes;
}
}
