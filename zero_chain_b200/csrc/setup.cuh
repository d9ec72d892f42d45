// Per-thread pieces of parameter generation (setup.cu) that the host emulation (tests/host_emul/emul_setup.cpp) compiles too:
// the signed-digit recoding and table walk of the batched fixed-base multiplication, the affine conversion with a shared
// inverse, and the segmented column sums of the QAP evaluation.
#pragma once
#include "curve.cuh"

namespace zksetup {

// ---- batched fixed-base multiplication ---------------------------------------------------------------------------------
// k g for many 256-bit k and one g: k = sum_w d_w 2^(C w) with signed digits |d_w| <= 2^(C-1), so with the table
// T[w][d - 1] = d 2^(C w) g (d = 1 .. 2^(C-1)) k g is one mixed addition per non-zero digit and no doubling.
// 256 / C + 1 windows: the last one takes the carry out of bit 255 (a full 256-bit k, not only k < r).
template <int C> struct FbGeom {
    static constexpr int W = 256 / C + 1;
    static constexpr int HALF = 1 << (C - 1);
    static constexpr int ENTRIES = W * HALF;
};
// digit of window w: bits [C w, C w + C) of k plus the carry of window w - 1, mapped to (-2^(C-1), 2^(C-1)]
template <int C>
ZK_DEV int fb_digit(const uint32_t *k, int w, uint32_t &carry) {
    const int lo = C * w;
    uint32_t v = 0;
    if (lo < 256) {
        const int i = lo >> 5, s = lo & 31;
        v = k[i] >> s;
        if (s + C > 32 && i + 1 < 8) v |= k[i + 1] << (32 - s);
        v &= (1u << C) - 1;
    }
    v += carry;
    if (v > (1u << (C - 1))) { carry = 1; return (int)v - (1 << C); }
    carry = 0;
    return (int)v;
}
// sum of the table points the digits of k select.  add_mixed is complete (P + P, P + (-P), infinity): for the windows at
// 2^255 and above a partial sum can equal +-the table point modulo r, and the base of zk_scalar_mul_many may be any point.
template <class F, int C>
ZK_DEV XYZZ<F> fb_walk(const Affine<F> *tbl, const uint32_t *k) {
    XYZZ<F> acc = XYZZ<F>::inf();
    uint32_t carry = 0;
#pragma unroll
    for (int w = 0; w < FbGeom<C>::W; w++) {
        const int d = fb_digit<C>(k, w, carry);
        if (d) {
            Affine<F> p = tbl[w * FbGeom<C>::HALF + (d < 0 ? -d : d) - 1];
            if (d < 0) p.y = p.y.neg();
            acc.add_mixed(p);
        }
    }
    return acc;
}
// d B for 1 <= d < 2^16 and an affine B, MSB-first (one table entry)
template <class F>
ZK_DEV XYZZ<F> fb_small_mul(const Affine<F> &b, uint32_t d) {
    int top = 15;
    while (top > 0 && !((d >> top) & 1)) top--;
    XYZZ<F> acc = XYZZ<F>::from_affine(b);
    for (int i = top - 1; i >= 0; i--) {
        acc = acc.dbl();
        if ((d >> i) & 1) acc.add_mixed(b);
    }
    return acc;
}
// affine conversion with a batch-shared inversion: each point contributes fb_denominator to a product over the batch, and
// gets back zzz_inv = 1 / its denominator (the inverse of the product times the other denominators).  Identities
// contribute 1 and come out as the all-zero affine pattern.
template <class F>
ZK_DEV F fb_denominator(const XYZZ<F> &q) { return q.is_inf() ? F::one() : q.zzz; }
template <class F>
ZK_DEV Affine<F> fb_affine(const XYZZ<F> &q, const F &zzz_inv) {
    if (q.is_inf()) return Affine<F>::inf();
    const F zi2 = (zzz_inv * q.zz).sqr();      // (ZZ / ZZZ)^2 = 1 / ZZ
    Affine<F> r; r.x = q.x * zi2; r.y = q.y * zzz_inv; return r;
}

// ---- QAP evaluation: segmented sums of the column-sorted matrix entries -------------------------------------------------
// After the counting sort by column, segment v (variable v) holds vals[seg_off[v] .. seg_off[v + 1]).  One pass cuts every
// segment into tasks of at most QAP_T entries (ceil(len / QAP_T) tasks, numbered by an exclusive scan into task_off) and sums
// each task, so no thread adds more than QAP_T values however skewed the columns are (the ONE variable sits in every boolean
// row of B).  The task sums are the next pass's segments; after ceil(log_QAP_T(max length)) passes each segment holds at most
// one value.
constexpr uint32_t QAP_T = 32;
ZK_DEV uint32_t qap_tasks_of(const uint32_t *seg_off, size_t v) { return (seg_off[v + 1] - seg_off[v] + QAP_T - 1) / QAP_T; }
// task t (< task_off[n_seg]): the sum of its entries
ZK_DEV Fr qap_task_sum(const uint32_t *seg_off, const uint32_t *task_off, size_t n_seg, const Fr *vals, uint32_t t) {
    size_t lo = 0, hi = n_seg;                  // last v with task_off[v] <= t: empty segments share their successor's offset
    while (hi - lo > 1) { size_t mid = (lo + hi) / 2; if (task_off[mid] <= t) lo = mid; else hi = mid; }
    const uint32_t b = seg_off[lo] + (t - task_off[lo]) * QAP_T, e0 = b + QAP_T, e = e0 < seg_off[lo + 1] ? e0 : seg_off[lo + 1];
    Fr acc = Fr::zero();
    for (uint32_t i = b; i < e; i++) acc = acc + vals[i];
    return acc;
}
ZK_DEV Fr qap_segment_value(const uint32_t *seg_off, const Fr *vals, size_t v) {
    return seg_off[v + 1] > seg_off[v] ? vals[seg_off[v]] : Fr::zero();
}

}  // namespace zksetup
