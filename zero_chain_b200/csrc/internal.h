// Shared host-side declarations of libzkb200 (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/zkb200.h"

void zk_set_error(const char *fmt, ...);
#define ZK_CUDA(call)                                                                                  \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            zk_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));       \
            return ZK_ERR_CUDA;                                                                        \
        }                                                                                              \
    } while (0)
#define ZK_TRY(call) do { int r__ = (call); if (r__ != ZK_OK) return r__; } while (0)

// grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return ZK_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes >> 3) + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { zk_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return ZK_ERR_CUDA; }
        cap = want;
        return ZK_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// one cached set of NTT twiddle tables (ntt.cu)
struct NttSlot { unsigned log_n = 0; bool valid = false; uint64_t last_use = 0; DevBuf w, g, gi, consts; };

// tuning options of a context (zk_ctx_set_opt); the prover lanes inherit them
struct zk_opts {
    long ba_min_entries = 1l << 22;    // ZK_OPT_AFFINE_MIN_ENTRIES; -1 = batched-affine rounds off
    long ba_levels = -1;               // ZK_OPT_AFFINE_LEVELS (-1 = from the average bucket length)
    long verify_lanes = 1;             // ZK_OPT_VERIFY_LANES: 1 = lane-parallel Miller loop / final exponentiation, 0 = thread per proof
};

struct zk_ctx {
    zk_opts opts;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    int *d_err = nullptr;          // device error flag (non-canonical scalar etc.)
    // MSM workspace
    DevBuf aff_pts0, aff_pts1, aff_scratch, aff_off0, aff_off1, aff_sizes0, aff_sizes1, aff_srcs, aff_tot;   // batched-affine rounds (msm_batchaff.cuh)
    DevBuf scalars, digits, tile_hist, tile_off, sizes, bucket_off, task_off, scan_scratch, sorted, partials, buckets, red_part, red_x, red_rows, sorted2, coarse_off, coarse_sizes, task_order, len_hist, heavy_list, red_tmp, result, out_bytes;
    bool len_hist_zeroed = false;
    // generic staging
    DevBuf stage_a, stage_b, stage_c;
    // NTT workspace + twiddle tables (per context: ordered on this context's stream, freed with it)
    DevBuf ntt_tmp;
    NttSlot ntt_slots[4];
    uint64_t ntt_clock = 0;
    bool ntt_attr_done = false;
    // groth16 workspace
    DevBuf g_a, g_b, g_c, g_h, g_scal, g_misc;
    // verifier workspace (pairing.cu)
    DevBuf v_pts, v_stat, v_coef, v_f, v_part, v_io;
    // live kernel timing (zk_ctx_profile): CUDA events around the dominant kernel on ctx->stream
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_events;   // pairs (start, stop)
    zk_ctx *aux2 = nullptr;        // third lane: the A MSM and s * g_a (independent of the NTT chain)
    zk_ctx *aux3 = nullptr;        // fourth lane: the B1 MSM and r * g_b1
    DevBuf g_scal3;                // A-query scalars
    zk_ctx *aux = nullptr;         // second lane (own stream + workspace) on the same device: the prover's G2 MSM overlaps the G1 work
    DevBuf g_scal2;                // B-query scalars (shared by the G1 and G2 B MSMs)
    DevBuf fb_tbl;                 // table of the batched fixed-base multiplication (setup.cu)
    // asynchronous MSM (zk_msm_begin / zk_msm_end): everything after the bucket accumulation runs on a HIGH-PRIORITY stream, so that
    // with two contexts in flight the latency-bound tail of one MSM is scheduled ahead of the other's accumulation blocks
    cudaStream_t tail = nullptr;
    cudaEvent_t ev_front = nullptr, ev_tail = nullptr;
    bool split_tail = false;       // set by zk_msm_*begin around the driver call
    size_t pending_bytes = 0;      // result bytes of the MSM in flight (0 = none)
    uint8_t *h_pinned = nullptr;   // small pinned buffer for results
    size_t h_pinned_cap = 0;
};

struct zk_bases {
    int group = 1;       // 1 = G1, 2 = G2
    int device = 0;
    size_t n = 0;        // bases (table row stride)
    int c = 0, W = 0;
    bool tables = false;
    void *d_tbl = nullptr;   // [W or 1][n] affine
};

int zk_use_device(zk_ctx *ctx);
// internal MSM driver: result XYZZ points (one per batch item) left in ctx->result (device)
int zk_msm_run(zk_ctx *ctx, const zk_bases *b, const void *d_scalars, size_t n, size_t batch);
int zk_encode_results(zk_ctx *ctx, int group, size_t count, int compressed, uint8_t *out_host);

// hot-TU entry points (msm_hot.cu)
int zk_msm_run_g1(zk_ctx *ctx, const zk_bases *b, const uint32_t *d_scalars, size_t n, size_t batch);
int zk_build_tables_g1(zk_ctx *ctx, zk_bases *b);
int zk_encode_results_g1(zk_ctx *ctx, size_t count, int compressed, uint8_t *d_out);
void zk_launch_bench_modmul(int field, int blocks, int threads, int iters, void *sink, cudaStream_t st);
int zk_bases_from_device(zk_ctx *ctx, int group, const void *d_points, size_t n, int window_bits, int precompute, zk_bases **out);
int zk_ntt_run(zk_ctx *ctx, void *d_data, unsigned log_n, int mode, size_t batch);
int zk_fr_load_evals(zk_ctx *ctx, const void *d_src, size_t n_c, unsigned log_m, int which, size_t batch, void *d_dst);
int zk_fr_quotient(zk_ctx *ctx, const void *d_abc, unsigned log_m, size_t batch, void *d_h);
int zk_fr_into_repr(zk_ctx *ctx, const void *d_h, unsigned log_m, size_t n_out, size_t n_total, size_t batch, void *d_scal);
int zk_fr_blinding_terms(zk_ctx *ctx, const void *d_r, const void *d_s, size_t batch, void *d_out);
int zk_check_err_flag(zk_ctx *ctx);
// lane-parallel verifier kernels (pairing_lanes.cu)
void zk_launch_miller_lanes(cudaStream_t st, size_t n, const void *a, const void *acc, const void *c, const void *coef_b, const void *gamma, int gamma_inf,
                            const void *delta, int delta_inf, const uint8_t *status, void *f);
void zk_launch_verify_final_lanes(cudaStream_t st, size_t n, const void *f, const void *alpha_beta, const uint8_t *status, uint8_t *verdict);
int zk_fr_to_mont(zk_ctx *ctx, const void *d_in, size_t n, void *d_out);
int zk_fr_witness_to_mont(zk_ctx *ctx, const void *d_inputs, size_t n_in, const void *d_aux, size_t n_aux, size_t batch, void *d_z);
// parameter generation and the batched fixed-base multiplication (setup.cu)
int zk_fixed_base(zk_ctx *ctx, int group, const void *d_base, const void *d_scalars, size_t n, void *d_out);
int zk_setup_powers(zk_ctx *ctx, const void *d_in, unsigned log_m, void *d_consts, int *d_flag, void *d_P, void *d_h);
int zk_setup_qap(zk_ctx *ctx, const uint32_t *d_row_ptr, const uint32_t *d_col, const void *d_coeff, size_t n_c, size_t nnz, size_t nv,
                 const void *d_L, size_t n_in_rows, uint32_t *scratch, void *d_vals0, void *d_vals1, void *d_out);
int zk_setup_flags(zk_ctx *ctx, const void *d_abc, const void *d_consts, size_t nv, size_t n_in, uint32_t *pos_a, uint32_t *pos_b, int *d_flag,
                   uint32_t *scratch);
int zk_setup_fill(zk_ctx *ctx, const void *d_abc, const void *d_consts, size_t nv, size_t n_in, const uint32_t *pos_a, const uint32_t *pos_b,
                  void *d_l, void *d_ic, void *d_a, void *d_b1, void *d_b2);
int zk_fr_r1cs_eval(zk_ctx *ctx, const uint32_t *d_row_ptr, const uint32_t *d_col, const void *d_coeff, const void *d_z, size_t n_c, size_t n_in,
                    size_t nv, unsigned log_m, int which, size_t batch, void *d_dst);
