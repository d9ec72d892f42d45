// libzkb200: execution context, MSM driver and diagnostics (host side of the C ABI, include/zkb200.h).
// The reference's counterpart is bellman's `multiexp` + `Worker` CPU pool (un-vendored, SURVEY.md §3.2);
// here the "pool" is one CUDA stream per context and the schedule documented in msm.cuh.
// Built "semi-hot" (field.cuh): the Fq product is inlined, the Fq2 product / square is the call boundary — the G2 MSM kernels of this
// translation unit run 10-20 % faster than with the Fq product as a function call, at 36 s of compile time.
#define ZK_SEMI_HOT 1
#include "internal.h"
#include "msm_driver.cuh"

using namespace zkmsm;

static thread_local char g_err[512] = "";
void zk_set_error(const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
extern "C" const char *zk_last_error(void) { return g_err; }
extern "C" const char *zk_version(void) { return "zkb200 0.1 (sm_100a)"; }
extern "C" int zk_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int zk_use_device(zk_ctx *ctx) { ZK_CUDA(cudaSetDevice(ctx->device)); return ZK_OK; }

extern "C" int zk_ctx_create(int device, void *stream, zk_ctx **out) {
    if (!out) { zk_set_error("zk_ctx_create: out is NULL"); return ZK_ERR_INVALID; }
    int n = zk_device_count();
    if (n == 0) { zk_set_error("no CUDA device: libzkb200 has no CPU fallback"); return ZK_ERR_CUDA; }
    if (device < 0 || device >= n) { zk_set_error("device %d out of range (%d devices)", device, n); return ZK_ERR_INVALID; }
    ZK_CUDA(cudaSetDevice(device));
    zk_ctx *c = new zk_ctx();
    c->device = device;
    if (stream) { c->stream = (cudaStream_t)stream; c->own_stream = false; }
    else { ZK_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }
    cudaDeviceProp prop;
    ZK_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    ZK_CUDA(cudaMalloc(&c->d_err, 32 * sizeof(int)));       // [0..1] error flags, [8..9] task length / heavy-bucket count, [10..17] work counters
    ZK_CUDA(cudaMemsetAsync(c->d_err, 0, 32 * sizeof(int), c->stream));
    c->h_pinned_cap = 1 << 20;
    ZK_CUDA(cudaMallocHost(&c->h_pinned, c->h_pinned_cap));
    *out = c;
    return ZK_OK;
}
extern "C" void zk_ctx_destroy(zk_ctx *c) {
    if (!c) return;
    if (c->aux) { zk_ctx_destroy(c->aux); c->aux = nullptr; }
    if (c->aux2) { zk_ctx_destroy(c->aux2); c->aux2 = nullptr; }
    if (c->aux3) { zk_ctx_destroy(c->aux3); c->aux3 = nullptr; }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    DevBuf *bufs[] = {&c->scalars, &c->digits, &c->tile_hist, &c->tile_off, &c->sizes, &c->bucket_off, &c->task_off, &c->scan_scratch,
                      &c->sorted, &c->partials, &c->buckets, &c->red_part, &c->red_x, &c->result, &c->out_bytes, &c->stage_a, &c->stage_b,
                      &c->stage_c, &c->ntt_tmp, &c->g_a, &c->g_b, &c->g_c, &c->g_h, &c->g_scal, &c->g_misc,
                      &c->aff_pts0, &c->aff_pts1, &c->aff_scratch, &c->aff_off0, &c->aff_off1, &c->aff_sizes0, &c->aff_sizes1, &c->aff_srcs, &c->aff_tot, &c->red_rows, &c->g_scal2, &c->g_scal3, &c->sorted2, &c->coarse_off, &c->coarse_sizes, &c->task_order, &c->len_hist, &c->heavy_list, &c->red_tmp,
                      &c->v_pts, &c->v_stat, &c->v_coef, &c->v_f, &c->v_part, &c->v_io, &c->fb_tbl};
    for (DevBuf *b : bufs) b->release();
    for (NttSlot &sl : c->ntt_slots) { sl.w.release(); sl.g.release(); sl.gi.release(); sl.consts.release(); }
    if (c->tail) { cudaStreamSynchronize(c->tail); cudaStreamDestroy(c->tail); cudaEventDestroy(c->ev_front); cudaEventDestroy(c->ev_tail); }
    if (c->d_err) cudaFree(c->d_err);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}
extern "C" int zk_ctx_set_opt(zk_ctx *c, int opt, long value) {
    if (!c) { zk_set_error("zk_ctx_set_opt: NULL ctx"); return ZK_ERR_INVALID; }
    for (zk_ctx *x : {c, c->aux, c->aux2, c->aux3}) {
        if (!x) continue;
        if (opt == ZK_OPT_AFFINE_MIN_ENTRIES) x->opts.ba_min_entries = value;
        else if (opt == ZK_OPT_AFFINE_LEVELS) x->opts.ba_levels = value;
        else if (opt == ZK_OPT_VERIFY_LANES) x->opts.verify_lanes = value;
        else { zk_set_error("zk_ctx_set_opt: unknown option %d", opt); return ZK_ERR_INVALID; }
    }
    return ZK_OK;
}
extern "C" int zk_ctx_sync(zk_ctx *c) { ZK_TRY(zk_use_device(c)); return zk_check_err_flag(c); }   // synchronises; reports a pending device-side error flag
extern "C" void *zk_ctx_stream(zk_ctx *c) { return (void *)c->stream; }

int zk_check_err_flag(zk_ctx *ctx) {
    int e[2] = {0, 0};
    ZK_CUDA(cudaMemcpyAsync(e, ctx->d_err, sizeof(e), cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    if (e[0] || e[1]) {
        ZK_CUDA(cudaMemsetAsync(ctx->d_err, 0, 2 * sizeof(int), ctx->stream));
        if (e[0]) { zk_set_error("scalar not canonical (>= r)"); return ZK_ERR_NOT_CANONICAL; }
        zk_set_error("point decoding failed (GroupDecodingError %d)", e[1]);
        return e[1] == zkcodec::DEC_INFINITY ? ZK_ERR_UNEXPECTED_IDENTITY : ZK_ERR_DECODE;
    }
    return ZK_OK;
}

// ---- bases ------------------------------------------------------------------------------------------
// Window size.  With precomputed tables all windows share one bucket set, so the cost is n * W mixed additions plus a
// reduction of 2^(c-1) buckets: 16 bits (W = 16, shared-memory one-level sort) up to 2^20 terms, 20 bits (W = 13,
// two-level sort) from 2^20 terms on — measured 7.7 ms vs 8.1 ms at 2^20.  17..19 bits are never picked: their top
// window holds only 8 / 3 / 0 scalar bits, which piles n/256 .. n entries into a few buckets.
static int pick_window(size_t n, bool tables) {
    int lg = 0;
    while (((size_t)1 << (lg + 1)) <= n) lg++;
    if (tables && lg >= 20) return 20;
    int c = lg - 1;
    if (c < 5) c = 5;
    if (c > 16) c = 16;
    return c;
}
__global__ void k_any_inf(const uint32_t *limbs, size_t n, int words, int *err) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t o = 0;
    for (int k = 0; k < words; k++) o |= limbs[i * words + k];
    if (!o) atomicCAS(err + 1, 0, zkcodec::DEC_INFINITY);
}
// device-resident variant used by the Groth16 CRS loader: d_points already holds n affine points
int zk_bases_from_device(zk_ctx *ctx, int group, const void *d_points, size_t n, int window_bits, int precompute, zk_bases **out) {
    if (group != 1 && group != 2) { zk_set_error("group must be 1 or 2"); return ZK_ERR_INVALID; }
    if (n == 0 || n >= ((size_t)1 << 27)) { zk_set_error("unsupported base count %zu", n); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    zk_bases *b = new zk_bases();
    b->group = group; b->device = ctx->device; b->n = n;
    b->c = window_bits > 0 ? window_bits : pick_window(n, precompute != 0);
    if (b->c < 2 || b->c > 20 || (b->c > 16 && !precompute)) { delete b; zk_set_error("window_bits must be in [2,16] (17..20 with precomputed tables)"); return ZK_ERR_INVALID; }
    b->W = 255 / b->c + 1;
    b->tables = precompute != 0;
    size_t psz = group == 1 ? sizeof(G1Affine) : sizeof(G2Affine);
    size_t rows = b->tables ? b->W : 1;
    cudaError_t e = cudaMalloc(&b->d_tbl, rows * n * psz);
    if (e != cudaSuccess) { delete b; zk_set_error("cudaMalloc tables (%zu B): %s", rows * n * psz, cudaGetErrorString(e)); return ZK_ERR_CUDA; }
    ZK_CUDA(cudaMemcpyAsync(b->d_tbl, d_points, n * psz, cudaMemcpyDeviceToDevice, ctx->stream));
    k_any_inf<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((const uint32_t *)b->d_tbl, n, (int)(psz / 4), ctx->d_err);
    int r = zk_check_err_flag(ctx);
    if (r) { zk_bases_free(b); return r; }
    if (b->tables) {
        r = group == 1 ? zk_build_tables_g1(ctx, b) : build_tables_t<Fq2>(ctx, b);
        if (r) { zk_bases_free(b); return r; }
    }
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = b;
    return ZK_OK;
}
extern "C" int zk_bases_upload(zk_ctx *ctx, int group, const uint64_t *limbs, size_t n, int window_bits, int precompute, zk_bases **out) {
    if (!ctx || !limbs || !out) { zk_set_error("zk_bases_upload: NULL argument"); return ZK_ERR_INVALID; }
    if (group != 1 && group != 2) { zk_set_error("group must be 1 or 2"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    size_t psz = group == 1 ? sizeof(G1Affine) : sizeof(G2Affine);
    ZK_TRY(ctx->stage_a.reserve(n * psz));
    ZK_CUDA(cudaMemcpyAsync(ctx->stage_a.p, limbs, n * psz, cudaMemcpyHostToDevice, ctx->stream));
    return zk_bases_from_device(ctx, group, ctx->stage_a.p, n, window_bits, precompute, out);
}
extern "C" void zk_bases_free(zk_bases *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->d_tbl) cudaFree(b->d_tbl);
    delete b;
}
extern "C" size_t zk_bases_len(const zk_bases *b) { return b ? b->n : 0; }
extern "C" int zk_bases_window_bits(const zk_bases *b) { return b ? b->c : 0; }

// ---- MSM driver: msm_driver.cuh, instantiated for G1 in msm_hot.cu and for G2 here ----
int zk_msm_run(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, size_t batch) {
    if (!ctx || !b || !d_scalars) { zk_set_error("zk_msm: NULL argument"); return ZK_ERR_INVALID; }
    if (b->device != ctx->device) { zk_set_error("bases live on device %d, context on %d", b->device, ctx->device); return ZK_ERR_INVALID; }
    if (n == 0 || batch == 0) { zk_set_error("empty MSM"); return ZK_ERR_INVALID; }
    if (b->tables ? n != b->n : n > b->n) {
        zk_set_error("scalar count %zu does not match the %zu bases (SynthesisError::AssignmentMissing)", n, b->n);
        return ZK_ERR_ASSIGNMENT_MISSING;
    }
    ZK_TRY(zk_use_device(ctx));
    return b->group == 1 ? zk_msm_run_g1(ctx, b, (const uint32_t *)d_scalars, n, batch) : msm_run_t<Fq2>(ctx, b, (const uint32_t *)d_scalars, n, batch);
}
int zk_encode_results(zk_ctx *ctx, int group, size_t count, int compressed, uint8_t *out_host) {
    size_t per = (group == 1 ? 96 : 192) / (compressed ? 2 : 1);
    ZK_TRY(ctx->out_bytes.reserve(count * per));
    if (count * per > ctx->h_pinned_cap) { zk_set_error("result batch too large"); return ZK_ERR_INVALID; }
    ZK_TRY(group == 1 ? zk_encode_results_g1(ctx, count, compressed, ctx->out_bytes.as<uint8_t>())
                      : encode_results_t<Fq2>(ctx, count, compressed, ctx->out_bytes.as<uint8_t>()));
    ZK_CUDA(cudaMemcpyAsync(ctx->h_pinned, ctx->out_bytes.p, count * per, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_TRY(zk_check_err_flag(ctx));   // synchronises the stream
    memcpy(out_host, ctx->h_pinned, count * per);
    return ZK_OK;
}
extern "C" int zk_msm_batch_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, size_t batch, uint8_t *out) {
    if (!out) { zk_set_error("zk_msm: out is NULL"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_msm_run(ctx, b, d_scalars, n, batch));
    return zk_encode_results(ctx, b->group, batch, 0, out);
}
extern "C" int zk_msm_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, uint8_t *out) {
    return zk_msm_batch_device(ctx, b, d_scalars, n, 1, out);
}
extern "C" int zk_msm(zk_ctx *ctx, const zk_bases *b, const uint64_t *scalars, size_t n, uint8_t *out) {
    if (!ctx || !scalars) { zk_set_error("zk_msm: NULL argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(ctx->scalars.reserve(n * 32));
    ZK_CUDA(cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    return zk_msm_device(ctx, b, ctx->scalars.p, n, out);
}
// one warp: out = sum of the n partial sums, each addition warp-cooperative (curve_coop.cuh)
template <class F>
__global__ void __launch_bounds__(32) k_fold_serial(const XYZZ<F> *in, int n, XYZZ<F> *out) {
    XYZZ<F> r = in[0];
    for (int i = 1; i < n; i++) zkcoop::add(r, in[i]);
    if (threadIdx.x == 0) out[0] = r;
}
// ---- asynchronous MSM: bellman's multiexp returns a future (multiexp.rs); begin / end is that future on CUDA streams ----
static const size_t PARTIAL_IN_FLIGHT = ~(size_t)0;      // pending_bytes sentinel: a partial MSM is in flight, no host result yet
static int ensure_tail(zk_ctx *ctx) {
    if (ctx->tail) return ZK_OK;
    int lo = 0, hi = 0;
    ZK_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    ZK_CUDA(cudaStreamCreateWithPriority(&ctx->tail, cudaStreamNonBlocking, hi));
    ZK_CUDA(cudaEventCreateWithFlags(&ctx->ev_front, cudaEventDisableTiming));
    ZK_CUDA(cudaEventCreateWithFlags(&ctx->ev_tail, cudaEventDisableTiming));
    return ZK_OK;
}
extern "C" void *zk_ctx_tail_stream(zk_ctx *ctx) {
    if (!ctx || zk_use_device(ctx) != ZK_OK || ensure_tail(ctx) != ZK_OK) return nullptr;
    return (void *)ctx->tail;
}
// affine conversion + wire format + D2H of ctx->result[0] on the tail stream; the context's stream is ordered after it
static int finish_on_tail(zk_ctx *ctx, int group) {
    const size_t per = group == 1 ? 96 : 192;
    ZK_TRY(ctx->out_bytes.reserve(per));
    cudaStream_t saved = ctx->stream;
    ctx->stream = ctx->tail;
    int r = group == 1 ? zk_encode_results_g1(ctx, 1, 0, ctx->out_bytes.as<uint8_t>()) : encode_results_t<Fq2>(ctx, 1, 0, ctx->out_bytes.as<uint8_t>());
    ctx->stream = saved;
    if (r) return r;
    ZK_CUDA(cudaMemcpyAsync(ctx->h_pinned, ctx->out_bytes.p, per, cudaMemcpyDeviceToHost, ctx->tail));
    ZK_CUDA(cudaEventRecord(ctx->ev_tail, ctx->tail));
    ZK_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_tail, 0));
    ctx->pending_bytes = per;
    return ZK_OK;
}
static int msm_split(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n) {
    ZK_TRY(ensure_tail(ctx));
    ctx->split_tail = true;
    int r = zk_msm_run(ctx, b, d_scalars, n, 1);
    ctx->split_tail = false;
    return r;
}
static int msm_begin_common(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n) {
    ZK_TRY(msm_split(ctx, b, d_scalars, n));
    return finish_on_tail(ctx, b->group);
}
// multi-GPU form of the future: the rank's partial sum (XYZZ, zk_partial_size bytes) is left in d_partial_out by the tail stream;
// the caller enqueues its all-gather on zk_ctx_tail_stream and then zk_points_fold_begin; zk_msm_end collects the folded result
extern "C" int zk_msm_partial_device_begin(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, void *d_partial_out) {
    if (!ctx || !b || !d_scalars || !d_partial_out) { zk_set_error("zk_msm_partial_device_begin: NULL argument"); return ZK_ERR_INVALID; }
    if (ctx->pending_bytes) { zk_set_error("zk_msm_partial_device_begin: an MSM is already in flight on this context"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(msm_split(ctx, b, d_scalars, n));
    ZK_CUDA(cudaMemcpyAsync(d_partial_out, ctx->result.p, zk_partial_size(b->group), cudaMemcpyDeviceToDevice, ctx->tail));
    ctx->pending_bytes = PARTIAL_IN_FLIGHT;
    return ZK_OK;
}
extern "C" int zk_points_fold_begin(zk_ctx *ctx, int group, const void *d_partials, size_t count) {
    if (!ctx || !d_partials || count == 0 || (group != 1 && group != 2)) { zk_set_error("zk_points_fold_begin: bad argument"); return ZK_ERR_INVALID; }
    if (ctx->pending_bytes && ctx->pending_bytes != PARTIAL_IN_FLIGHT) { zk_set_error("zk_points_fold_begin: a result is already pending on this context"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(ensure_tail(ctx));
    ZK_TRY(ctx->result.reserve(4 * sizeof(G2XYZZ)));
    if (group == 1) k_fold_serial<Fq><<<1, 32, 0, ctx->tail>>>((const G1XYZZ *)d_partials, (int)count, ctx->result.as<G1XYZZ>());
    else k_fold_serial<Fq2><<<1, 32, 0, ctx->tail>>>((const G2XYZZ *)d_partials, (int)count, ctx->result.as<G2XYZZ>());
    ZK_CUDA(cudaGetLastError());
    ctx->pending_bytes = 0;
    return finish_on_tail(ctx, group);
}
extern "C" int zk_msm_device_begin(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n) {
    if (!ctx || !b || !d_scalars) { zk_set_error("zk_msm_device_begin: NULL argument"); return ZK_ERR_INVALID; }
    if (ctx->pending_bytes) { zk_set_error("zk_msm_device_begin: an MSM is already in flight on this context (call zk_msm_end first)"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    return msm_begin_common(ctx, b, d_scalars, n);
}
extern "C" int zk_msm_begin(zk_ctx *ctx, const zk_bases *b, const uint64_t *scalars, size_t n) {
    if (!ctx || !b || !scalars) { zk_set_error("zk_msm_begin: NULL argument"); return ZK_ERR_INVALID; }
    if (ctx->pending_bytes) { zk_set_error("zk_msm_begin: an MSM is already in flight on this context (call zk_msm_end first)"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(ctx->scalars.reserve(n * 32));
    ZK_CUDA(cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    return msm_begin_common(ctx, b, ctx->scalars.p, n);
}
extern "C" int zk_msm_end(zk_ctx *ctx, uint8_t *out) {
    if (!ctx || !out) { zk_set_error("zk_msm_end: NULL argument"); return ZK_ERR_INVALID; }
    if (!ctx->pending_bytes || ctx->pending_bytes == PARTIAL_IN_FLIGHT) { zk_set_error("zk_msm_end: no result in flight"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    size_t per = ctx->pending_bytes;
    ctx->pending_bytes = 0;
    ZK_CUDA(cudaEventSynchronize(ctx->ev_tail));
    ZK_TRY(zk_check_err_flag(ctx));
    memcpy(out, ctx->h_pinned, per);
    return ZK_OK;
}
extern "C" size_t zk_partial_size(int group) { return group == 1 ? sizeof(G1XYZZ) : sizeof(G2XYZZ); }
extern "C" int zk_msm_partial_device(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, void *d_partial_out) {
    if (!d_partial_out) { zk_set_error("zk_msm_partial_device: out is NULL"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_msm_run(ctx, b, d_scalars, n, 1));
    ZK_CUDA(cudaMemcpyAsync(d_partial_out, ctx->result.p, zk_partial_size(b->group), cudaMemcpyDeviceToDevice, ctx->stream));
    return zk_check_err_flag(ctx);
}
extern "C" int zk_points_fold(zk_ctx *ctx, int group, const void *d_partials, size_t count, uint8_t *out) {
    if (!ctx || !d_partials || !out || count == 0) { zk_set_error("zk_points_fold: bad argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(ctx->result.reserve(4 * sizeof(G2XYZZ)));
    if (group == 1) k_fold_serial<Fq><<<1, 32, 0, ctx->stream>>>((const G1XYZZ *)d_partials, (int)count, ctx->result.as<G1XYZZ>());
    else k_fold_serial<Fq2><<<1, 32, 0, ctx->stream>>>((const G2XYZZ *)d_partials, (int)count, ctx->result.as<G2XYZZ>());
    ZK_CUDA(cudaGetLastError());
    return zk_encode_results(ctx, group, 1, 0, out);
}

// ---- utilities -----------------------------------------------------------------------------------------------
#ifdef ZK_EXPERIMENTS
// the previous path, one thread per point with a full double-and-add; experiment builds select it with ZK_FB_OLD=1 so that
// tools/setup_bench.py can compare the two on the same scalars
template <class F>
__global__ void __launch_bounds__(128) k_scalar_mul_many(const Affine<F> *base, const uint32_t *scalars, size_t n, Affine<F> *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k[8];
    for (int j = 0; j < 8; j++) k[j] = scalars[i * 8 + j];
    out[i] = scalar_mul(XYZZ<F>::from_affine(base[0]), k).to_affine();
}
#endif
// the batched fixed-base multiplication of parameter generation (setup.cu): any 256-bit scalar, exact k * base
extern "C" int zk_scalar_mul_many(zk_ctx *ctx, int group, const uint64_t *base, const uint64_t *scalars, size_t n, uint64_t *out) {
    if (!ctx || !base || !scalars || !out) { zk_set_error("zk_scalar_mul_many: NULL argument"); return ZK_ERR_INVALID; }
    if (group != 1 && group != 2) { zk_set_error("group must be 1 or 2"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    size_t psz = group == 1 ? sizeof(G1Affine) : sizeof(G2Affine);
    ZK_TRY(ctx->stage_a.reserve(psz)); ZK_TRY(ctx->stage_b.reserve(n * 32)); ZK_TRY(ctx->stage_c.reserve(n * psz));
    ZK_CUDA(cudaMemcpyAsync(ctx->stage_a.p, base, psz, cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(cudaMemcpyAsync(ctx->stage_b.p, scalars, n * 32, cudaMemcpyHostToDevice, ctx->stream));
#ifdef ZK_EXPERIMENTS
    if (getenv("ZK_FB_OLD") && atoi(getenv("ZK_FB_OLD")) && n) {
        unsigned blk = (unsigned)((n + 127) / 128);
        if (group == 1) k_scalar_mul_many<Fq><<<blk, 128, 0, ctx->stream>>>(ctx->stage_a.as<G1Affine>(), ctx->stage_b.as<uint32_t>(), n, ctx->stage_c.as<G1Affine>());
        else k_scalar_mul_many<Fq2><<<blk, 128, 0, ctx->stream>>>(ctx->stage_a.as<G2Affine>(), ctx->stage_b.as<uint32_t>(), n, ctx->stage_c.as<G2Affine>());
        ZK_CUDA(cudaGetLastError());
    } else
#endif
    ZK_TRY(zk_fixed_base(ctx, group, ctx->stage_a.p, ctx->stage_b.p, n, ctx->stage_c.p));
    ZK_CUDA(cudaMemcpyAsync(out, ctx->stage_c.p, n * psz, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZK_OK;
}

template <class T>
__global__ void k_field_op(int op, const T *a, const T *b, size_t n, T *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T x = a[i], y = b ? b[i] : x, r;
    switch (op) {
    case 0: r = x * y; break;
    case 1: r = x + y; break;
    case 2: r = x - y; break;
    case 3: r = x.sqr(); break;
    case 4: r = x.inverse(); break;
    case 5: r = T::canonical_lt_mod(x) ? T::from_canonical(x) : T::zero(); break;
    default: r = x.to_canonical(); break;
    }
    out[i] = r;
}
extern "C" int zk_field_op(zk_ctx *ctx, int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out) {
    if (!ctx || !a || !out || op < 0 || op > 6 || (field != 0 && field != 1)) { zk_set_error("zk_field_op: bad argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    size_t sz = field == 0 ? 48 : 32;
    ZK_TRY(ctx->stage_a.reserve(n * sz)); ZK_TRY(ctx->stage_b.reserve(n * sz)); ZK_TRY(ctx->stage_c.reserve(n * sz));
    ZK_CUDA(cudaMemcpyAsync(ctx->stage_a.p, a, n * sz, cudaMemcpyHostToDevice, ctx->stream));
    if (b) ZK_CUDA(cudaMemcpyAsync(ctx->stage_b.p, b, n * sz, cudaMemcpyHostToDevice, ctx->stream));
    unsigned blk = (unsigned)((n + 127) / 128);
    if (field == 0) k_field_op<Fq><<<blk, 128, 0, ctx->stream>>>(op, ctx->stage_a.as<Fq>(), b ? ctx->stage_b.as<Fq>() : nullptr, n, ctx->stage_c.as<Fq>());
    else k_field_op<Fr><<<blk, 128, 0, ctx->stream>>>(op, ctx->stage_a.as<Fr>(), b ? ctx->stage_b.as<Fr>() : nullptr, n, ctx->stage_c.as<Fr>());
    ZK_CUDA(cudaGetLastError());
    ZK_CUDA(cudaMemcpyAsync(out, ctx->stage_c.p, n * sz, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZK_OK;
}

extern "C" int zk_bench_modmul(zk_ctx *ctx, int field, int blocks, int threads, int iters, double *per_s, double *ms_out) {
    if (!ctx || !per_s) { zk_set_error("zk_bench_modmul: NULL argument"); return ZK_ERR_INVALID; }
#ifndef ZK_EXPERIMENTS
    if (field != 0 && field != 1) { zk_set_error("zk_bench_modmul: field must be 0 (Fq) or 1 (Fr)"); return ZK_ERR_INVALID; }
#endif
    ZK_TRY(zk_use_device(ctx));
    ZK_TRY(ctx->stage_a.reserve(64));
    cudaEvent_t e0, e1;
    ZK_CUDA(cudaEventCreate(&e0)); ZK_CUDA(cudaEventCreate(&e1));
    for (int rep = 0; rep < 2; rep++) {
        ZK_CUDA(cudaEventRecord(e0, ctx->stream));
        zk_launch_bench_modmul(field, blocks, threads, iters, ctx->stage_a.p, ctx->stream);
        ZK_CUDA(cudaEventRecord(e1, ctx->stream));
        ZK_CUDA(cudaEventSynchronize(e1));
    }
    float ms = 0;
    ZK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *per_s = (double)blocks * threads * iters * 4.0 / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    return ZK_OK;
}

// ---- live kernel timing -----------------------------------------------------------------------------------
extern "C" int zk_ctx_profile(zk_ctx *ctx, int enable) {
    if (!ctx) { zk_set_error("zk_ctx_profile: NULL ctx"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    for (cudaEvent_t ev : ctx->prof_events) cudaEventDestroy(ev);
    ctx->prof_events.clear();
    ctx->prof_on = enable != 0;
    for (zk_ctx *c : {ctx, ctx->aux, ctx->aux2, ctx->aux3})  // work counters of this context and its lanes restart with the profile
        if (c) { ZK_CUDA(cudaStreamSynchronize(c->stream)); ZK_CUDA(cudaMemsetAsync(c->d_err + 10, 0, 8 * sizeof(int), c->stream)); ZK_CUDA(cudaStreamSynchronize(c->stream)); }
    return ZK_OK;
}
extern "C" int zk_ctx_profile_counts(zk_ctx *ctx, uint64_t *g1_additions, uint64_t *g2_additions, uint64_t *g1_xyzz, uint64_t *g2_xyzz) {
    if (!ctx || !g1_additions || !g2_additions || !g1_xyzz || !g2_xyzz) { zk_set_error("zk_ctx_profile_counts: NULL argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    *g1_additions = 0; *g2_additions = 0; *g1_xyzz = 0; *g2_xyzz = 0;
    for (zk_ctx *c : {ctx, ctx->aux, ctx->aux2, ctx->aux3}) {
        if (!c) continue;
        unsigned long long v[4] = {0, 0, 0, 0};
        ZK_CUDA(cudaStreamSynchronize(c->stream));
        if (c->tail) ZK_CUDA(cudaStreamSynchronize(c->tail));
        ZK_CUDA(cudaMemcpy(v, c->d_err + 10, sizeof(v), cudaMemcpyDeviceToHost));
        *g1_additions += v[0]; *g2_additions += v[1]; *g1_xyzz += v[2]; *g2_xyzz += v[3];     // ints 10-11, 12-13, 14-15, 16-17 of d_err
    }
    return ZK_OK;
}
extern "C" int zk_ctx_profile_read(zk_ctx *ctx, double *total_ms, uint64_t *launches) {
    if (!ctx || !total_ms || !launches) { zk_set_error("zk_ctx_profile_read: NULL argument"); return ZK_ERR_INVALID; }
    ZK_TRY(zk_use_device(ctx));
    ZK_CUDA(cudaStreamSynchronize(ctx->stream));
    double tot = 0;
    for (size_t i = 0; i + 1 < ctx->prof_events.size(); i += 2) {
        float ms = 0;
        ZK_CUDA(cudaEventElapsedTime(&ms, ctx->prof_events[i], ctx->prof_events[i + 1]));
        tot += ms;
    }
    *total_ms = tot;
    *launches = ctx->prof_events.size() / 2;
    return ZK_OK;
}
