// C ABI of libadapted_b200.so (see include/adapted_b200.h).  Single translation unit: the kernels live in the
// .cuh files included below.  Build: adapted_b200/csrc/build.py (nvcc -gencode arch=compute_100a,code=sm_100a).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/adapted_b200.h"
#include "adb_common.cuh"
#include "adb_ctx.cuh"
#include "adb_global.cuh"
#include "adb_gsample.cuh"
#include "adb_llr.cuh"
#include "adb_read_kernel.cuh"
#include "adb_cnn.cuh"
#include "adb_stream.cuh"
#include "adb_stream_session.cuh"
#include "adb_cnn_tc.cuh"
#include "adb_vhist.cuh"
#include "adb_start_peak.cuh"
#include "adb_legacy.cuh"

extern "C" int adb_abi_version(void) { return ADB_ABI_VERSION; }
extern "C" const char *adb_last_error(void) { return adb_err_string().c_str(); }
extern "C" int adb_record_size(void) { return (int)sizeof(adb_record); }
extern "C" int adb_config_size(void) { return (int)sizeof(adb_config); }
extern "C" int adb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// slots of the constant bank adb_c_convT (adb_cnn.cuh): one per live context and device, -1 when none is left (the
// context then keeps the transposed convolution's weights in shared memory)
static std::mutex g_ct_mu;
static unsigned g_ct_used[64];
static int ct_slot_take(int device) {
    std::lock_guard<std::mutex> lk(g_ct_mu);
    if (device < 0 || device >= 64) return -1;
    for (int s = 0; s < ADB_CT_SLOTS; s++)
        if (!(g_ct_used[device] & (1u << s))) { g_ct_used[device] |= 1u << s; return s; }
    return -1;
}
static void ct_slot_give(int device, int slot) {
    std::lock_guard<std::mutex> lk(g_ct_mu);
    if (device >= 0 && device < 64 && slot >= 0) g_ct_used[device] &= ~(1u << slot);
}

extern "C" int adb_ctx_create(int device, adb_ctx **out) {
    if (!out) return ADB_ERR_ARG;
    *out = nullptr;
    int n = adb_device_count();
    if (n <= 0) {
        set_err("no CUDA device available: adapted_b200 has no CPU fallback");
        return ADB_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        set_err("invalid device index");
        return ADB_ERR_ARG;
    }
    CUDA_TRY(cudaSetDevice(device));
    adb_ctx *c = new adb_ctx();
    c->device = device;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (const char *e = getenv("ADB_HIST_VALIDATE")) c->opt_hist_validate = atoi(e);  // A/B switch of the validation kernel
    c->ct_slot = ct_slot_take(device);
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) {
        CUDA_TRY(cudaEventCreateWithFlags(&c->p_done[k], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->p_copied[k], cudaEventDisableTiming));
    }
    *out = c;
    return ADB_OK;
}

extern "C" int adb_ctx_set_timing(adb_ctx *c, int on);
extern "C" void adb_ctx_destroy(adb_ctx *c) {
    if (!c) return;
    if (c->twin) { adb_ctx_destroy(c->twin); c->twin = nullptr; }
    cudaSetDevice(c->device);
    ct_slot_give(c->device, c->ct_slot);
    c->ct_slot = -1;
    if (c->file_ring && c->file_ring_free) { c->file_ring_free(c->file_ring); c->file_ring = nullptr; }
    DevBuf *all[] = {&c->states, &c->hist, &c->series, &c->given, &c->status, &c->cnn_x, &c->cnn_act0,
                     &c->cnn_act1, &c->cnn_scores, &c->cnn_w, &c->cnn_aux, &c->cnn_post, &c->sp_rows, &c->h_signal, &c->h_offsets,
                     &c->h_lens, &c->h_coff, &c->h_cscale, &c->h_records, &c->h_misc, &c->h_misc2, &c->h_misc3,
                     &c->gsb_plan, &c->gsb_hist, &c->gsb_tab, &c->gsb_bases, &c->gsb_active, &c->vf_done, &c->mvs_perm, &c->cnn_wtc, &c->cnn_a0t, &c->cnn_ct, &c->llr_cc, &c->val_cc, &c->z_fail};
    for (DevBuf *b : all) b->release();
    for (int k = 0; k < 2; k++) {
        DevBuf *pb[] = {&c->p_signal[k], &c->p_offsets[k], &c->p_lens[k], &c->p_coff[k], &c->p_cscale[k], &c->p_records[k], &c->p_status[k],
                        &c->p_comp[k], &c->p_coffs[k], &c->p_nsamp[k], &c->p_frames[k], &c->p_foffs[k], &c->p_zstat[k]};
        for (DevBuf *b : pb) b->release();
        if (c->p_done[k]) cudaEventDestroy(c->p_done[k]);
        if (c->p_copied[k]) cudaEventDestroy(c->p_copied[k]);
    }
    adb_ctx_set_timing(c, 0);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int64_t adb_ctx_launch_count(const adb_ctx *c) { return c ? c->launches : 0; }

extern "C" int adb_ctx_set_option(adb_ctx *c, const char *name, int value) {
    if (!c || !name) return ADB_ERR_ARG;
    if (!strcmp(name, "exact_global_select")) { c->opt_exact_gsel = value; return ADB_OK; }
    if (!strcmp(name, "no_fast_validate")) { c->opt_no_fast_validate = value; return ADB_OK; }
    if (!strcmp(name, "hist_validate")) { c->opt_hist_validate = value; return ADB_OK; }
    if (!strcmp(name, "cnn_fp32_pipe")) { c->opt_cnn_fp32 = value; return ADB_OK; }
    if (!strcmp(name, "pipeline_copy_only")) { c->opt_copy_only = value; return ADB_OK; }
    if (!strcmp(name, "no_cand_followup")) { c->opt_no_cand_followup = value; return ADB_OK; }
    if (!strcmp(name, "host_zstd")) { c->opt_host_zstd = value; return ADB_OK; }
    set_err(std::string("unknown option: ") + name);
    return ADB_ERR_ARG;
}

// diagnostics of the most recent call on this context (synchronises the context's stream)
extern "C" int64_t adb_ctx_query(adb_ctx *c, const char *name) {
    if (!c || !name) return -1;
    if (!strcmp(name, "global_select_fallbacks")) {
        // minibatches of the last LLR call that the sampled select handed to the exact multi-pass select
        if (!c->gsb_last_batches || !c->gsb_active.p) return 0;
        std::vector<int> h(c->gsb_last_batches);
        if (cudaSetDevice(c->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(h.data(), c->gsb_active.p, sizeof(int) * h.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t n = 0;
        for (int v : h) n += (v != 0);
        return n;
    }
    if (!strcmp(name, "validate_handovers")) {
        // reads of the last pass that validate_fast_kernel left to validate_kernel
        if (!c->vf_last_reads || !c->vf_done.p) return 0;
        std::vector<unsigned char> h(c->vf_last_reads);
        if (cudaSetDevice(c->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(h.data(), c->vf_done.p, h.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t n = 0;
        for (unsigned char v : h) n += (v == 0);
        return n;
    }
    if (!strcmp(name, "zstd_host_frames")) return c->zstd_host_frames;
    return -1;
}

extern "C" int adb_ctx_set_timing(adb_ctx *c, int on) {
    if (!c) return ADB_ERR_ARG;
    c->timing = on;
    for (int k = 0; k < 8; k++) {
        for (auto &p : c->ev[k]) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
        c->ev[k].clear();
        c->timing_ms[k] = 0;
        c->timing_n[k] = 0;
    }
    return ADB_OK;
}

// out[16] = {ms, launches} for the 8 kernel classes; call after the stream has been synchronised
extern "C" int adb_ctx_get_timing(adb_ctx *c, double *out) {
    if (!c || !out) return ADB_ERR_ARG;
    for (int k = 0; k < 8; k++) {
        for (auto &p : c->ev[k]) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) { c->timing_ms[k] += ms; c->timing_n[k] += 1; }
            cudaEventDestroy(p.first);
            cudaEventDestroy(p.second);
        }
        c->ev[k].clear();
        out[2 * k] = c->timing_ms[k];
        out[2 * k + 1] = (double)c->timing_n[k];
    }
    return ADB_OK;
}

static BatchDev to_dev_view(const adb_batch &b) {
    BatchDev d;
    d.signal = b.signal;
    d.sig_type = b.sig_type;
    d.n_reads = b.n_reads;
    d.m = b.m;
    d.batch_size = b.batch_size;
    d.offsets = b.offsets;
    d.full_lens = b.full_lens;
    d.calib_offset = b.calib_offset;
    d.calib_scale = b.calib_scale;
    return d;
}

static int check_batch(const adb_batch *b) {
    if (!b || !b->signal || !b->full_lens || b->n_reads < 0 || b->m <= 0 || b->batch_size <= 0) {
        set_err("invalid adb_batch");
        return ADB_ERR_ARG;
    }
    if (b->sig_type == ADB_SIG_I16 && (!b->offsets || !b->calib_offset || !b->calib_scale)) {
        set_err("ADB_SIG_I16 needs offsets and calibration");
        return ADB_ERR_ARG;
    }
    if (b->sig_type != ADB_SIG_I16 && b->sig_type != ADB_SIG_F32) {
        set_err("unknown sig_type");
        return ADB_ERR_ARG;
    }
    return ADB_OK;
}

static int check_config(const adb_config *cfg) {
    if (!cfg) return ADB_ERR_ARG;
    if (cfg->mvs_detect_check && cfg->mvs_detect_overwrite) {
        // mean_var_shift_polyA_detect_at_loc reads moving_*[2 * offset] (mvs.py:289-290): an IndexError in the
        // reference when the search window is not longer than the larger moving window
        const int offset = cfg->pA_mean_window > cfg->pA_var_window ? cfg->pA_mean_window : cfg->pA_var_window;
        if (cfg->search_window <= offset || cfg->search_window < 1) {
            set_err("mvs_detect_overwrite needs search_window > max(pA_mean_window, pA_var_window)");
            return ADB_ERR_UNSUPPORTED;
        }
    }
    if (cfg->downscale_factor < 1 || cfg->downscale_factor > 128 || cfg->sp_downscale_factor < 1 ||
        cfg->sp_downscale_factor > 128) {
        set_err("downscale_factor must be in [1, 128]");
        return ADB_ERR_UNSUPPORTED;
    }
    if (cfg->mean_window < 1 || cfg->mean_window > ADB_MAX_MEAN_WINDOW || cfg->pA_var_window > ADB_MAX_MOVE_WINDOW ||
        cfg->pA_mean_window > ADB_MAX_MOVE_WINDOW || cfg->pA_var_window < 1 || cfg->pA_mean_window < 1) {
        set_err("window sizes outside the supported range");
        return ADB_ERR_UNSUPPORTED;
    }
    if (cfg->polya_cand_k > ADB_MAX_CAND) {
        set_err("polya_cand_k exceeds ADB_MAX_CAND");
        return ADB_ERR_UNSUPPORTED;
    }
    return ADB_OK;
}

// ---- global median / MAD -------------------------------------------------------------------------------------
// int16 sources: sampled one-pass select (adb_gsample.cuh); whatever it cannot settle -- and every float32 source --
// goes through the exact multi-pass radix select (adb_global.cuh), whose kernels skip the settled minibatches.
static int run_global_med_mad(adb_ctx *ctx, const BatchDev &B, int n_batches, int max_obs_trace, cudaStream_t st) {
    if (ctx->states.ensure(sizeof(GselState) * (size_t)n_batches)) { set_err("cudaMalloc states"); return ADB_ERR_CUDA; }
    if (ctx->hist.ensure(sizeof(unsigned) * 2 * GSEL_BINS * (size_t)n_batches)) { set_err("cudaMalloc hist"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemsetAsync(ctx->states.p, 0, sizeof(GselState) * (size_t)n_batches, st));
    CUDA_TRY(cudaMemsetAsync(ctx->hist.p, 0, sizeof(unsigned) * 2 * GSEL_BINS * (size_t)n_batches, st));
    const int gx = std::max(1, std::min(B.batch_size, (ctx->sm_count * 8 + n_batches - 1) / n_batches));
    const int *active = nullptr;
    ctx->gsb_last_batches = 0;
    if (B.sig_type == ADB_SIG_I16 && !ctx->opt_exact_gsel) {
        if (ctx->gsb_plan.ensure(sizeof(GsbPlan) * (size_t)n_batches) || ctx->gsb_hist.ensure(sizeof(unsigned) * GSB_BINS * (size_t)n_batches) ||
            ctx->gsb_tab.ensure(sizeof(unsigned) * GSB_TAB * (size_t)B.n_reads) || ctx->gsb_bases.ensure(sizeof(GsbRead) * (size_t)B.n_reads) ||
            ctx->gsb_active.ensure(sizeof(int) * (size_t)n_batches)) { set_err("cudaMalloc sampled select"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemsetAsync(ctx->gsb_hist.p, 0, sizeof(unsigned) * GSB_BINS * (size_t)n_batches, st));
        CUDA_TRY(cudaMemsetAsync(ctx->gsb_tab.p, 0, sizeof(unsigned) * GSB_TAB * (size_t)B.n_reads, st));
        const size_t sm = sizeof(unsigned) * GSB_BINS;
        CUDA_TRY(cudaFuncSetAttribute(gsb_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        CUDA_TRY(cudaFuncSetAttribute(gsb_plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        const int gs = std::max(1, std::min(B.batch_size, (ctx->sm_count * 3 + n_batches - 1) / n_batches));
        {
            KernelTimer t(ctx, 1, st);
            // about GSB_TARGET_SAMPLE samples per minibatch, never denser than every 4th sample
            const long long per_mb = (long long)std::min(B.batch_size, B.n_reads) * std::max(1, std::min(max_obs_trace, B.m));
            const int stride = (int)std::max<long long>(4, std::min<long long>(GSB_STRIDE, per_mb / GSB_TARGET_SAMPLE));
            gsb_sample_kernel<<<dim3(gs, n_batches), 256, sm, st>>>(B, max_obs_trace, stride, (unsigned *)ctx->gsb_hist.p);
            gsb_plan_kernel<<<n_batches, 256, sm, st>>>((const unsigned *)ctx->gsb_hist.p, (GsbPlan *)ctx->gsb_plan.p);
        }
        {
            KernelTimer t(ctx, 0, st);
            gsb_pass_kernel<<<dim3(gx, n_batches), 256, 0, st>>>(B, max_obs_trace, (GsbPlan *)ctx->gsb_plan.p,
                                                                 (unsigned *)ctx->gsb_tab.p, (GsbRead *)ctx->gsb_bases.p);
        }
        {
            KernelTimer t(ctx, 1, st);
            gsb_finish_kernel<<<n_batches, 256, 0, st>>>(B, (GsbPlan *)ctx->gsb_plan.p, (const unsigned *)ctx->gsb_tab.p,
                                                         (const GsbRead *)ctx->gsb_bases.p, (GselState *)ctx->states.p,
                                                         (int *)ctx->gsb_active.p);
        }
        ctx->launches += 4;
        ctx->gsb_last_batches = n_batches;
        active = (const int *)ctx->gsb_active.p;
    }
    dim3 grid(gx, n_batches);
    for (int stage = 0; stage < 2; stage++) {
        for (int pass = 0; pass < 3; pass++) {
            {
                KernelTimer t(ctx, active ? 7 : 0, st);
                gsel_hist_kernel<<<grid, 256, 0, st>>>(B, max_obs_trace, stage, pass, (const GselState *)ctx->states.p,
                                                       (unsigned *)ctx->hist.p, active);
            }
            {
                KernelTimer t(ctx, active ? 7 : 1, st);
                gsel_scan_kernel<<<n_batches, 256, 0, st>>>(stage, pass, (GselState *)ctx->states.p, (unsigned *)ctx->hist.p, active);
            }
            ctx->launches += 2;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

__global__ void merge_status_kernel(const GselState *states, int *batch_status, int n_batches) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_batches) {
        int s = states[i].status;
        if (s != ADB_OK) atomicMin(&batch_status[i], s);
    }
}

// ---- the detect entry point (device pointers) -----------------------------------------------------------------
static int trace_dims(const adb_config &cfg, int span, int *nds_max, int *peak_cap) {
    *nds_max = std::max(64, (std::max(span, 0) + cfg.downscale_factor - 1) / cfg.downscale_factor + 2);
    *peak_cap = *nds_max / 2 + 24;  // >= 16 slots per 32-position chunk of cta_peaks_prepare
    return 0;
}

static int launch_llr_primary(adb_ctx *ctx, const BatchDev &B, const adb_config &cfg, int *given, int *ntopk,
                              int *batch_status, cudaStream_t st) {
    PrimaryArgs A;
    A.B = B;
    A.gstates = (const GselState *)ctx->states.p;
    trace_dims(cfg, cfg.max_obs_trace - cfg.min_obs_adapter, &A.nds_max, &A.peak_cap);
    A.given = given;
    A.ntopk = ntopk;
    A.batch_status = batch_status;
    size_t smem = trace_smem_bytes(A.nds_max, A.peak_cap, true);
    if ((int)smem > ctx->max_smem_optin) {
        set_err("downscaled LLR trace of llr_primary_kernel does not fit in shared memory (max_obs_trace / downscale_factor too large)");
        return ADB_ERR_UNSUPPORTED;
    }
    CUDA_TRY(cudaFuncSetAttribute(llr_primary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, llr_primary_kernel, ADB_TRACE_THREADS, smem));
    if (occ < 1) occ = 1;
    int grid = std::max(1, std::min(B.n_reads, ctx->sm_count * occ));
    // the prefix sums of the read a CTA works on: 2 x nds_max doubles per CTA in global memory
    if (ctx->llr_cc.ensure(sizeof(double) * 2 * (size_t)A.nds_max * (size_t)grid)) { set_err("cudaMalloc llr prefix sums"); return ADB_ERR_CUDA; }
    A.cc = (double *)ctx->llr_cc.p;
    {
        KernelTimer t(ctx, 3, st);
        llr_primary_kernel<<<grid, ADB_TRACE_THREADS, smem, st>>>(A, cfg);
    }
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

static int launch_validate(adb_ctx *ctx, const BatchDev &B, const adb_config &cfg, int mode, const int *given,
                           int given_stride, int given_ntopk, const int *ntopk_per_read, adb_record *out,
                           const int *batch_status, cudaStream_t st) {
    ValidateArgs A;
    A.B = B;
    A.given = given;
    A.given_stride = given_stride;
    A.given_ntopk = given_ntopk;
    A.ntopk_per_read = ntopk_per_read;
    A.mode = mode;
    A.win_bytes = B.m * (B.sig_type == ADB_SIG_F32 ? 4 : 2);
    A.nds_max = 0;
    A.peak_cap = 0;
    if (mode == ADB_METHOD_CNN && cfg.fallback_to_llr_short_reads) trace_dims(cfg, B.m, &A.nds_max, &A.peak_cap);
    A.out = out;
    A.batch_status = batch_status;
    A.hm_cc = nullptr;
    // the read's window staged in shared memory where it fits next to the scratch; longer windows are read from global
    // memory (win_bytes = 0), and the hail-mary trace keeps its prefix sums in global memory (a third of the
    // trace's shared memory, so that several CTAs share an SM)
    const bool staged = validate_smem_bytes(A.win_bytes, A.nds_max, A.peak_cap) <= (size_t)ctx->max_smem_optin;
    if (!staged) A.win_bytes = 0;
    const bool hm_ext = !staged && A.nds_max > 0;
    const size_t smem = validate_smem_bytes(A.win_bytes, A.nds_max, A.peak_cap, hm_ext);
    if (smem > (size_t)ctx->max_smem_optin) {
        set_err("hail-mary trace of validate_kernel does not fit in shared memory (sig_preload_size / downscale_factor too large)");
        return ADB_ERR_UNSUPPORTED;
    }
    CUDA_TRY(cudaFuncSetAttribute(validate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, validate_kernel, ADB_VAL_THREADS, smem));
    if (occ < 1) occ = 1;
    // moving statistics of the first poly(A) candidate are precomputed thread-per-read into compact pools sized for
    // an average poly(A) share of 1/4 of the window; reads that do not fit fall back to the in-CTA path (same result)
    const bool overwrite = cfg.mvs_detect_check && cfg.mvs_detect_overwrite;  // general kernel only (row f3)
    const bool pre = cfg.mvs_detect_check != 0 && !overwrite;
    // Pool sized for the worst case -- every read's poly(A) candidate at the end of the window (the long-poly(A) stress
    // set gets close, and rows are handed out longest first, so a pool that is too small starves the many short rows)
    // -- as far as a third of the free device memory allows; an ordinary job touches about a tenth of it.
    long long pool_cap = std::max<long long>(1 << 20, (long long)B.n_reads * B.m);
    if ((size_t)pool_cap * sizeof(float) * 2 > ctx->cnn_aux.cap) {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
            const long long budget = (long long)((free_b + ctx->cnn_aux.cap) / 3 / (2 * sizeof(float)));
            pool_cap = std::max<long long>(std::min<long long>(pool_cap, budget), std::max<long long>(1 << 20, (long long)B.n_reads * B.m / 4));
        }
    }
    pool_cap &= ~3LL;  // the second pool starts pool_cap floats behind the first: rows stay 16-byte aligned in both
    if (pre && (ctx->cnn_aux.ensure((size_t)pool_cap * sizeof(float) * 2) ||
                ctx->h_misc3.ensure(sizeof(int) * 2 * (size_t)B.n_reads + sizeof(long long) * ((size_t)B.n_reads + 2) + sizeof(float) * 2 * (size_t)B.n_reads))) {
        set_err("cudaMalloc moving-statistics scratch");
        return ADB_ERR_CUDA;
    }
    int grid_max = std::max(1, ctx->sm_count * occ);
    const size_t row = (size_t)B.m * sizeof(float);
    if (ctx->series.ensure((size_t)grid_max * 2 * row)) { set_err("cudaMalloc series"); return ADB_ERR_CUDA; }
    A.series = (float *)ctx->series.p;
    if (hm_ext) {
        if (ctx->val_cc.ensure(sizeof(double) * 2 * (size_t)A.nds_max * (size_t)grid_max)) { set_err("cudaMalloc hail-mary prefix sums"); return ADB_ERR_CUDA; }
        A.hm_cc = (double *)ctx->val_cc.p;
    }
    A.pre_var = A.pre_mean = nullptr;
    A.pre_off = nullptr;
    A.pre_meta = nullptr;
    const float *series_med = nullptr;
    if (pre) {
        MvsSeriesArgs M;
        M.B = B;
        M.given = given;
        M.given_stride = given_stride;
        M.n_reads = B.n_reads;
        M.var_pool = (float *)ctx->cnn_aux.p;
        M.mean_pool = M.var_pool + pool_cap;
        M.pool_cap = pool_cap;
        long long *lbase = (long long *)ctx->h_misc3.p;
        M.cursor = (unsigned long long *)lbase;
        M.row_off = lbase + 2;
        M.meta = (int *)(lbase + 2 + B.n_reads);
        CUDA_TRY(cudaMemsetAsync(M.cursor, 0, 16, st));
        M.perm = nullptr;
        M.n_active = nullptr; M.all_cands = 0; M.n_cand = given_ntopk; M.ntopk_per_read = ntopk_per_read;
        {
            KernelTimer t(ctx, 4, st);
            if (B.sig_type == ADB_SIG_I16) {
                // reads of similar segment length share a warp (counting sort by length, three tiny kernels)
                if (ctx->mvs_perm.ensure(sizeof(int) * ((size_t)B.n_reads + MVS_NBUCKET))) { set_err("cudaMalloc mvs perm"); return ADB_ERR_CUDA; }
                int *bucket = (int *)ctx->mvs_perm.p, *perm = bucket + MVS_NBUCKET;
                CUDA_TRY(cudaMemsetAsync(bucket, 0, sizeof(int) * MVS_NBUCKET, st));
                const int sgrid = std::max(1, std::min((B.n_reads + 255) / 256, ctx->sm_count * 4));
                mvs_len_hist_kernel<<<sgrid, 256, 0, st>>>(M, cfg, bucket);
                mvs_len_scan_kernel<<<1, MVS_NBUCKET, 0, st>>>(bucket);
                mvs_len_scatter_kernel<<<sgrid, 256, 0, st>>>(M, cfg, bucket, perm);
                ctx->launches += 3;
                M.perm = perm;
                CUDA_TRY(cudaFuncSetAttribute(mvs_series_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mvs_smem_bytes()));
                mvs_series_kernel<<<(B.n_reads + MVS_LANES - 1) / MVS_LANES, MVS_LANES, mvs_smem_bytes(), st>>>(M, cfg);
                if (!ctx->opt_no_fast_validate) {
                    // medians of the two series of every row, one warp per series (consumed by validate_fast_kernel)
                    SeriesMedianArgs SM;
                    SM.B = B; SM.pre_var = M.var_pool; SM.pre_mean = M.mean_pool; SM.pre_off = M.row_off; SM.pre_meta = M.meta;
                    SM.perm = perm; SM.n_reads = B.n_reads;
                    SM.out = (float *)(M.meta + 2 * (size_t)B.n_reads);
                    series_med = SM.out;
                    const size_t ssm = series_median_smem_bytes();
                    CUDA_TRY(cudaFuncSetAttribute(series_median_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
                    int socc = 0;
                    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&socc, series_median_kernel, SM_WARPS * 32, ssm));
                    const int sgrid2 = std::max(1, std::min((2 * B.n_reads + SM_WARPS - 1) / SM_WARPS, ctx->sm_count * std::max(socc, 1)));
                    series_median_kernel<<<sgrid2, SM_WARPS * 32, ssm, st>>>(SM, cfg);
                    ctx->launches += 1;
                }
            } else {
                mvs_series_f32_kernel<<<(B.n_reads + 127) / 128, 128, 0, st>>>(M, cfg);
            }
        }
        ctx->launches += 1;
        A.pre_var = M.var_pool;
        A.pre_mean = M.mean_pool;
        A.pre_off = M.row_off;
        A.pre_meta = M.meta;
    }
    A.done = nullptr;
    A.pending = A.n_pending = nullptr;
    A.work_counter = nullptr;
    ctx->vf_last_reads = 0;
    if (B.sig_type == ADB_SIG_I16 && !ctx->opt_no_fast_validate && !overwrite) {
        // int16 sources: counting-based validation (adb_vfast.cuh); what it leaves is picked up by validate_kernel.
        // It stages the window (dynamic shared memory) next to its static scratch: both count against the limit.
        const size_t fsm = vfast_smem_bytes(B.m * 2);
        cudaFuncAttributes fa, ca;
        CUDA_TRY(cudaFuncGetAttributes(&fa, validate_fast_kernel));
        CUDA_TRY(cudaFuncGetAttributes(&ca, validate_cand_kernel));
        if (fsm + std::max(fa.sharedSizeBytes, ca.sharedSizeBytes) <= (size_t)ctx->max_smem_optin) {
            if (ctx->vf_done.ensure((size_t)B.n_reads + 16)) { set_err("cudaMalloc done flags"); return ADB_ERR_CUDA; }
            CUDA_TRY(cudaMemsetAsync(ctx->vf_done.p, 0, (size_t)B.n_reads + 16, st));
            VfastArgs F;
            F.B = B; F.given = given; F.given_stride = given_stride; F.given_ntopk = given_ntopk; F.ntopk_per_read = ntopk_per_read;
            F.mode = mode; F.win_bytes = B.m * 2; F.out = out; F.batch_status = batch_status;
            F.pre_var = A.pre_var; F.pre_mean = A.pre_mean; F.pre_off = A.pre_off; F.pre_meta = A.pre_meta;
            F.series_med = series_med;
            F.done = (unsigned char *)ctx->vf_done.p;
            F.cand_followup = (pre && mode == ADB_METHOD_CNN && (ntopk_per_read || given_ntopk > 1) && !ctx->opt_no_cand_followup) ? 1 : 0;
            CUDA_TRY(cudaFuncSetAttribute(validate_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm));
            int focc = 0;
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&focc, validate_fast_kernel, VF_THREADS, fsm));
            if (focc < 1) focc = 1;
            const int fgrid = std::max(1, std::min(B.n_reads, ctx->sm_count * focc));
            // the tensor-core histogram variant needs an accumulator per piece of the window: the ranges of the MVS check
            // and of the median-shift check together can cut a read into more pieces than it has
            const bool use_hist = ctx->opt_hist_validate && B.m <= 65535 && !(cfg.mvs_detect_check && cfg.detect_med_shift);
            if (use_hist) {
                const size_t hsm = vhist_smem_bytes();
                CUDA_TRY(cudaFuncSetAttribute(validate_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsm));
                // Four CTAs per SM: 128 of the SM's 512 TMEM columns, 64 registers x 256 threads and ~45 KB of shared memory
                // each.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for a kernel that allocates tensor
                // memory; the CTAs do run side by side: 88.7 / 48.6 / 28.9 ms at 1 / 2 / 4 CTAs per SM.)
                int hocc = 4;
                if (const char *e = getenv("ADB_HIST_OCC")) hocc = std::max(1, std::min(atoi(e), 4));
                const int hgrid = std::max(1, std::min(B.n_reads, ctx->sm_count * hocc));
                if (getenv("ADB_DEBUG_OCC")) fprintf(stderr, "validate_hist_kernel: occupancy %d, grid %d, smem %zu\n", hocc, hgrid, hsm);
                KernelTimer t(ctx, 2, st);
                validate_hist_kernel<<<hgrid, VF_THREADS, hsm, st>>>(F, cfg);
            } else {
                KernelTimer t(ctx, 2, st);
                validate_fast_kernel<<<fgrid, VF_THREADS, fsm, st>>>(F, cfg);
            }
            ctx->launches += 1;
            A.done = F.done;
            ctx->vf_last_reads = B.n_reads;
            if (pre && mode == ADB_METHOD_CNN && (ntopk_per_read || given_ntopk > 1)) {
                // what is left mostly failed its first poly(A) candidate: the general kernel walks further candidates
                // (and the hail-mary end), each needing the two moving-statistics series.  One thread-per-read pass
                // up to the largest candidate serves them all as prefixes (the pools of the first pass are free now).
                MvsSeriesArgs M;
                M.B = B; M.given = given; M.given_stride = given_stride; M.n_reads = B.n_reads;
                M.var_pool = (float *)A.pre_var; M.mean_pool = (float *)A.pre_mean; M.pool_cap = pool_cap;
                long long *lbase = (long long *)ctx->h_misc3.p;
                M.cursor = (unsigned long long *)lbase;
                M.row_off = lbase + 2;
                M.meta = (int *)(lbase + 2 + B.n_reads);
                int *cnt = (int *)ctx->mvs_perm.p, *list = cnt + MVS_NBUCKET;  // counting-sort scratch of the first pass
                CUDA_TRY(cudaMemsetAsync(M.cursor, 0, 16, st));
                CUDA_TRY(cudaMemsetAsync(cnt, 0, 2 * sizeof(int), st));  // [0] list length, [1] work counter of validate_kernel
                A.pending = list; A.n_pending = cnt; A.work_counter = cnt + 1;
                M.perm = list; M.n_active = cnt; M.all_cands = 1; M.n_cand = given_ntopk; M.ntopk_per_read = ntopk_per_read;
                KernelTimer t(ctx, 7, st);
                mvs_pending_kernel<<<(B.n_reads + 255) / 256, 256, 0, st>>>(F.done, B.n_reads, list, cnt);
                mvs_series_kernel<<<(B.n_reads + MVS_LANES - 1) / MVS_LANES, MVS_LANES, mvs_smem_bytes(), st>>>(M, cfg);
                ctx->launches += 2;
                if (F.cand_followup) {
                    // the further candidates of the reads whose first one failed, from the rows of the pass above
                    VfastArgs F2 = F;
                    F2.pre_var = M.var_pool; F2.pre_mean = M.mean_pool; F2.pre_off = M.row_off; F2.pre_meta = M.meta;
                    CUDA_TRY(cudaFuncSetAttribute(validate_cand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm));
                    validate_cand_kernel<<<fgrid, VF_THREADS, fsm, st>>>(F2, cfg, list, cnt);
                    ctx->launches += 1;
                }
            }
        }
    }
    {
        int grid = std::max(1, std::min(B.n_reads, grid_max));
        KernelTimer t(ctx, A.done ? 7 : 2, st);
        validate_kernel<<<grid, ADB_VAL_THREADS, smem, st>>>(A, cfg);
    }
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

// minibatches processed by one set of launches: bounds the scratch arena (moving-statistics pools, tallies, CNN
// activations) for calls of any size; larger calls are cut at minibatch boundaries, which never changes a record
#define ADB_MAX_BATCHES_PER_PASS 256

static int detect_dev_pass(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                           adb_record *out_records, int32_t *batch_status, cudaStream_t st);

extern "C" int adb_detect_dev(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                              adb_record *out_records, int32_t *batch_status, void *cuda_stream) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    if (batch->n_reads == 0) return ADB_OK;
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    for (int b0 = 0; b0 < n_batches; b0 += ADB_MAX_BATCHES_PER_PASS) {
        const int r0 = b0 * batch->batch_size;
        const int r1 = (int)std::min<long long>((long long)(b0 + ADB_MAX_BATCHES_PER_PASS) * batch->batch_size, batch->n_reads);
        adb_batch sub = *batch;
        sub.n_reads = r1 - r0;
        sub.full_lens = batch->full_lens + r0;
        if (batch->sig_type == ADB_SIG_F32) {
            sub.signal = (const float *)batch->signal + (size_t)r0 * batch->m;
        } else {  // offsets stay absolute: the blob pointer does not move
            sub.offsets = batch->offsets + r0;
            sub.calib_offset = batch->calib_offset + r0;
            sub.calib_scale = batch->calib_scale + r0;
        }
        rc = detect_dev_pass(ctx, &sub, cfg, cnn_weights, out_records + r0, batch_status ? batch_status + b0 : nullptr, st);
        if (rc) return rc;
    }
    return ADB_OK;
}

static int detect_dev_pass(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                           adb_record *out_records, int32_t *batch_status, cudaStream_t st) {
    int rc = ADB_OK;
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    BatchDev B = to_dev_view(*batch);
    int *status = batch_status;
    if (!status) {
        if (ctx->status.ensure(sizeof(int) * (size_t)n_batches)) { set_err("cudaMalloc status"); return ADB_ERR_CUDA; }
        status = (int *)ctx->status.p;
    }
    CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(int) * (size_t)n_batches, st));
    if (cfg->primary_method == ADB_METHOD_LLR) {
        rc = run_global_med_mad(ctx, B, n_batches, cfg->max_obs_trace, st);
        if (rc) return rc;
        merge_status_kernel<<<(n_batches + 127) / 128, 128, 0, st>>>((const GselState *)ctx->states.p, status, n_batches);
        ctx->launches += 1;
        if (ctx->given.ensure(sizeof(int) * (size_t)batch->n_reads * 3)) { set_err("cudaMalloc given"); return ADB_ERR_CUDA; }
        int *given = (int *)ctx->given.p, *ntopk = given + (size_t)batch->n_reads * 2;
        rc = launch_llr_primary(ctx, B, *cfg, given, ntopk, status, st);
        if (rc) return rc;
        return launch_validate(ctx, B, *cfg, ADB_METHOD_LLR, given, 2, -1, ntopk, out_records, status, st);
    } else if (cfg->primary_method == ADB_METHOD_CNN) {
        if (!cnn_weights) { set_err("cnn_weights required for the CNN primary method"); return ADB_ERR_ARG; }
        const int stride = 1 + std::max(1, cfg->polya_cand_k);
        if (ctx->given.ensure(sizeof(int) * (size_t)batch->n_reads * stride)) { set_err("cudaMalloc given"); return ADB_ERR_CUDA; }
        rc = cnn_primary_boundaries(ctx, B, *cfg, cnn_weights, (int *)ctx->given.p, st);
        if (rc) return rc;
        return launch_validate(ctx, B, *cfg, ADB_METHOD_CNN, (const int *)ctx->given.p, stride,
                               std::max(1, cfg->polya_cand_k), nullptr, out_records, status, st);
    } else if (cfg->primary_method == ADB_METHOD_START_PEAK) {
        if (ctx->given.ensure(sizeof(int) * (size_t)batch->n_reads * 2)) { set_err("cudaMalloc given"); return ADB_ERR_CUDA; }
        rc = start_peak_primary(ctx, B, *cfg, (int *)ctx->given.p, out_records, status, st);
        if (rc) return rc;
        rc = launch_validate(ctx, B, *cfg, ADB_METHOD_START_PEAK, (const int *)ctx->given.p, 2, -1, nullptr, out_records, status, st);
        if (rc) return rc;
        return start_peak_finish(ctx, B, *cfg, out_records, st);
    }
    set_err("unknown primary_method");
    return ADB_ERR_ARG;
}

// ---- host-buffer convenience wrappers ------------------------------------------------------------------------------
// Error paths of the *_host entry points: asynchronous copies into / out of the CALLER's buffers may still be in
// flight when a later step fails; the streams are drained before the status is returned, so the caller may free its
// buffers as soon as the call is back.
struct StreamDrain {
    cudaStream_t s[4] = {nullptr, nullptr, nullptr, nullptr};
    int n = 0;
    bool armed = true;
    void add(cudaStream_t st) { if (st && n < 4) s[n++] = st; }
    ~StreamDrain() {
        if (!armed) return;
        for (int i = 0; i < n; i++) cudaStreamSynchronize(s[i]);
    }
};

struct StagedBatch {
    adb_batch dev;
    size_t signal_bytes;
};

static int stage_batch(adb_ctx *ctx, const adb_batch *b, StagedBatch *out, cudaStream_t st) {
    adb_batch d = *b;
    size_t sig_bytes;
    if (b->sig_type == ADB_SIG_F32) sig_bytes = (size_t)b->n_reads * b->m * sizeof(float);
    else sig_bytes = (size_t)b->offsets[b->n_reads] * sizeof(int16_t);
    if (ctx->h_signal.ensure(sig_bytes + 64)) { set_err("cudaMalloc signal staging"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(ctx->h_signal.p, b->signal, sig_bytes, cudaMemcpyHostToDevice, st));
    d.signal = ctx->h_signal.p;
    if (ctx->h_lens.ensure(sizeof(int32_t) * (size_t)b->n_reads + 16)) { set_err("cudaMalloc lens"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(ctx->h_lens.p, b->full_lens, sizeof(int32_t) * (size_t)b->n_reads, cudaMemcpyHostToDevice, st));
    d.full_lens = (const int32_t *)ctx->h_lens.p;
    if (b->sig_type == ADB_SIG_I16) {
        if (ctx->h_offsets.ensure(sizeof(int64_t) * ((size_t)b->n_reads + 1)) || ctx->h_coff.ensure(sizeof(float) * (size_t)b->n_reads + 16) ||
            ctx->h_cscale.ensure(sizeof(float) * (size_t)b->n_reads + 16)) { set_err("cudaMalloc staging"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemcpyAsync(ctx->h_offsets.p, b->offsets, sizeof(int64_t) * ((size_t)b->n_reads + 1), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ctx->h_coff.p, b->calib_offset, sizeof(float) * (size_t)b->n_reads, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ctx->h_cscale.p, b->calib_scale, sizeof(float) * (size_t)b->n_reads, cudaMemcpyHostToDevice, st));
        d.offsets = (const int64_t *)ctx->h_offsets.p;
        d.calib_offset = (const float *)ctx->h_coff.p;
        d.calib_scale = (const float *)ctx->h_cscale.p;
    } else {
        d.offsets = nullptr;
        d.calib_offset = d.calib_scale = nullptr;
    }
    out->dev = d;
    out->signal_bytes = sig_bytes;
    return ADB_OK;
}

extern "C" int adb_detect_host(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                               adb_record *out_records, int32_t *batch_status) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (batch->n_reads == 0) return ADB_OK;
    cudaStream_t st = ctx->stream;
    StreamDrain drain;
    drain.add(st);
    StagedBatch sb;
    rc = stage_batch(ctx, batch, &sb, st);
    if (rc) return rc;
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    if (ctx->h_records.ensure(sizeof(adb_record) * (size_t)batch->n_reads)) { set_err("cudaMalloc records"); return ADB_ERR_CUDA; }
    if (ctx->h_misc.ensure(sizeof(int) * (size_t)n_batches + 16)) { set_err("cudaMalloc status"); return ADB_ERR_CUDA; }
    const float *w_dev = nullptr;
    if (cnn_weights && cfg->primary_method == ADB_METHOD_CNN) {
        if (ctx->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc weights"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemcpyAsync(ctx->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, st));
        w_dev = (const float *)ctx->h_misc2.p;
    }
    rc = adb_detect_dev(ctx, &sb.dev, cfg, w_dev, (adb_record *)ctx->h_records.p, (int *)ctx->h_misc.p, st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_records, ctx->h_records.p, sizeof(adb_record) * (size_t)batch->n_reads, cudaMemcpyDeviceToHost, st));
    if (batch_status)
        CUDA_TRY(cudaMemcpyAsync(batch_status, ctx->h_misc.p, sizeof(int) * (size_t)n_batches, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// Pipelined ingest for long jobs: the reads are cut into chunks of `chunk_batches` minibatches; the H2D copy of
// chunk i+1 (copy stream) overlaps the kernels of chunk i (compute stream), records return per chunk.  Host buffers
// should be pinned (cudaHostAlloc / torch pin_memory) for the copies to be asynchronous.  I16 ragged input only.
extern "C" int adb_detect_pipelined_host(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg,
                                         const float *cnn_weights, adb_record *out_records, int32_t *batch_status,
                                         int32_t chunk_batches) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    if (batch->sig_type != ADB_SIG_I16) { set_err("pipelined ingest takes ragged int16 input"); return ADB_ERR_ARG; }
    if (chunk_batches < 1) chunk_batches = 1;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (batch->n_reads == 0) return ADB_OK;
    const float *w_dev = nullptr;
    if (cfg->primary_method == ADB_METHOD_CNN) {
        if (!cnn_weights) { set_err("cnn_weights required"); return ADB_ERR_ARG; }
        if (ctx->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc weights"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemcpyAsync(ctx->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, ctx->stream));
        w_dev = (const float *)ctx->h_misc2.p;
    }
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    // Chunk schedule (in minibatches).  The first copy and the last chunk's kernels cannot overlap anything, so the
    // job starts and ends with small chunks (chunk_batches / 4, / 2) and runs full-size chunks in between, where the
    // per-chunk launch overheads and kernel tails matter.
    std::vector<int> sched;
    {
        const int q = std::max(1, chunk_batches / 4), h = std::max(1, chunk_batches / 2);
        int left = n_batches;
        std::vector<int> tail;
        if (n_batches >= 2 * (q + h) + chunk_batches) {
            sched.push_back(q); sched.push_back(h);
            tail.push_back(h); tail.push_back(q);
            left -= 2 * (q + h);
        }
        while (left > 0) { const int c = std::min(left, chunk_batches); sched.push_back(c); left -= c; }
        sched.insert(sched.end(), tail.begin(), tail.end());
    }
    // consecutive chunks alternate between this context and its twin: each has its own compute stream and scratch arena,
    // the copies of all chunks go through one copy stream in order
    if (!ctx->twin && sched.size() >= 3) {
        rc = adb_ctx_create(ctx->device, &ctx->twin);
        if (rc) return rc;
    }
    if (ctx->twin) {
        ctx->twin->opt_no_fast_validate = ctx->opt_no_fast_validate;
        ctx->twin->opt_hist_validate = ctx->opt_hist_validate;
        ctx->twin->opt_cnn_fp32 = ctx->opt_cnn_fp32;
        ctx->twin->opt_exact_gsel = ctx->opt_exact_gsel;
        ctx->twin->opt_no_cand_followup = ctx->opt_no_cand_followup;
    }
    adb_ctx *cc[2] = {ctx, ctx->twin ? ctx->twin : ctx};
    const float *w_devs[2] = {w_dev, w_dev};
    if (w_dev && ctx->twin) {
        if (ctx->twin->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc weights"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemcpyAsync(ctx->twin->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, ctx->twin->stream));
        w_devs[1] = (const float *)ctx->twin->h_misc2.p;
    }
    cudaStream_t cs = ctx->copy_stream;
    StreamDrain drain;
    drain.add(cs);
    drain.add(ctx->stream);
    if (ctx->twin) drain.add(ctx->twin->stream);
    int b0 = 0;  // first minibatch of the chunk
    for (int ch = 0; ch < (int)sched.size(); ch++) {
        adb_ctx *c = cc[ch & 1];
        const int slot = ctx->twin ? 0 : (ch & 1);
        cudaStream_t ks = c->stream;
        const int r0 = b0 * batch->batch_size;
        const int r1 = (int)std::min<long long>((long long)batch->n_reads, (long long)(b0 + sched[ch]) * batch->batch_size), nr = r1 - r0;
        const int nb = (nr + batch->batch_size - 1) / batch->batch_size;
        const int64_t e0 = batch->offsets[r0], e1 = batch->offsets[r1];
        // the slot is free once the D2H of the chunk that used it two iterations ago has finished
        if (ch >= 2) CUDA_TRY(cudaEventSynchronize(c->p_done[slot]));
        if (c->p_signal[slot].ensure((size_t)(e1 - e0) * 2 + 64) || c->p_offsets[slot].ensure(sizeof(int64_t) * ((size_t)nr + 1)) ||
            c->p_lens[slot].ensure(sizeof(int32_t) * (size_t)nr + 16) || c->p_coff[slot].ensure(sizeof(float) * (size_t)nr + 16) ||
            c->p_cscale[slot].ensure(sizeof(float) * (size_t)nr + 16) || c->p_records[slot].ensure(sizeof(adb_record) * (size_t)nr) ||
            c->p_status[slot].ensure(sizeof(int) * (size_t)nb + 16)) { set_err("cudaMalloc pipeline staging"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemcpyAsync(c->p_signal[slot].p, (const int16_t *)batch->signal + e0, (size_t)(e1 - e0) * 2, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_offsets[slot].p, batch->offsets + r0, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_lens[slot].p, batch->full_lens + r0, sizeof(int32_t) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_coff[slot].p, batch->calib_offset + r0, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_cscale[slot].p, batch->calib_scale + r0, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaEventRecord(c->p_copied[slot], cs));
        CUDA_TRY(cudaStreamWaitEvent(ks, c->p_copied[slot], 0));
        adb_batch d = *batch;
        // offsets stay absolute: rebase the blob pointer so that blob[offsets[i]] is the staged copy
        d.signal = (const int16_t *)c->p_signal[slot].p - e0;
        d.offsets = (const int64_t *)c->p_offsets[slot].p;
        d.full_lens = (const int32_t *)c->p_lens[slot].p;
        d.calib_offset = (const float *)c->p_coff[slot].p;
        d.calib_scale = (const float *)c->p_cscale[slot].p;
        d.n_reads = nr;
        if (!ctx->opt_copy_only) {
            rc = adb_detect_dev(c, &d, cfg, w_devs[ch & 1], (adb_record *)c->p_records[slot].p, (int *)c->p_status[slot].p, ks);
            if (rc) return rc;
        }
        CUDA_TRY(cudaMemcpyAsync(out_records + r0, c->p_records[slot].p, sizeof(adb_record) * (size_t)nr, cudaMemcpyDeviceToHost, ks));
        if (batch_status)
            CUDA_TRY(cudaMemcpyAsync(batch_status + b0, c->p_status[slot].p, sizeof(int) * (size_t)nb, cudaMemcpyDeviceToHost, ks));
        CUDA_TRY(cudaEventRecord(c->p_done[slot], ks));
        b0 += sched[ch];
    }
    if (ctx->twin) CUDA_TRY(cudaStreamSynchronize(ctx->twin->stream));
    cudaStream_t ks = ctx->stream;
    CUDA_TRY(cudaStreamSynchronize(ks));
    CUDA_TRY(cudaStreamSynchronize(cs));
    return ADB_OK;
}

extern "C" int adb_global_med_mad_host(adb_ctx *ctx, const adb_batch *batch, int32_t max_obs_trace, float *med_mad) {
    if (!ctx || !med_mad) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StagedBatch sb;
    rc = stage_batch(ctx, batch, &sb, st);
    if (rc) return rc;
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    rc = run_global_med_mad(ctx, to_dev_view(sb.dev), n_batches, max_obs_trace, st);
    if (rc) return rc;
    std::vector<GselState> hs(n_batches);
    CUDA_TRY(cudaMemcpyAsync(hs.data(), ctx->states.p, sizeof(GselState) * (size_t)n_batches, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < n_batches; i++) { med_mad[2 * i] = hs[i].med; med_mad[2 * i + 1] = hs[i].mad; }
    return ADB_OK;
}

// ---- streaming poly(A) detector (row f4) ----------------------------------------------------------------------------
static int check_stream_config(const adb_stream_config *cfg) {
    if (cfg->pA_mean_window < 1 || cfg->pA_var_window < 1 || cfg->pA_mean_window > ADB_MAX_MOVE_WINDOW ||
        cfg->pA_var_window > ADB_MAX_MOVE_WINDOW || cfg->min_obs_adapter < 0 || cfg->search_increment_step < 1 ||
        cfg->polyA_window < 1 || cfg->median_shift_window < 1) {
        set_err("streaming config outside the supported range");
        return ADB_ERR_UNSUPPORTED;
    }
    return ADB_OK;
}

extern "C" int adb_mvs_stream_detect_host(adb_ctx *ctx, const adb_batch *batch, const adb_stream_config *cfg,
                                          int32_t *polya_start) {
    if (!ctx || !cfg || !polya_start) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    rc = check_stream_config(cfg);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (batch->n_reads == 0) return ADB_OK;
    cudaStream_t st = ctx->stream;
    StagedBatch sb;
    rc = stage_batch(ctx, batch, &sb, st);
    if (rc) return rc;
    StreamArgs A;
    A.B = to_dev_view(sb.dev);
    A.win_bytes = A.B.m * (A.B.sig_type == ADB_SIG_F32 ? 4 : 2);
    const size_t smem = (((size_t)A.win_bytes + 48 + 15) & ~(size_t)15) + (((size_t)ADB_SEL_SMEM_BYTES + 64 + 15) & ~(size_t)15) + 256;
    if ((int)smem > ctx->max_smem_optin) { set_err("signal window does not fit in shared memory"); return ADB_ERR_UNSUPPORTED; }
    CUDA_TRY(cudaFuncSetAttribute(mvs_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mvs_stream_kernel, ADB_VAL_THREADS, smem));
    if (occ < 1) occ = 1;
    const int grid = std::max(1, std::min(A.B.n_reads, ctx->sm_count * occ));
    if (ctx->series.ensure((size_t)grid * 2 * (size_t)A.B.m * sizeof(float)) ||
        ctx->h_misc.ensure(sizeof(int32_t) * (size_t)A.B.n_reads + 16)) { set_err("cudaMalloc stream scratch"); return ADB_ERR_CUDA; }
    A.series = (float *)ctx->series.p;
    A.out = (int32_t *)ctx->h_misc.p;
    mvs_stream_kernel<<<grid, ADB_VAL_THREADS, smem, st>>>(A, *cfg);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(polya_start, A.out, sizeof(int32_t) * (size_t)A.B.n_reads, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- read-until sessions of the streaming detector (adb_stream_session.cuh) ---------------------------------------
struct adb_stream_session {
    adb_ctx *ctx = nullptr;
    adb_stream_config cfg;
    bool f32 = false;  // the caches hold calibrated float32 pA (else int16 ADC codes)
    bool dev = false;  // pushes come from device memory (adb_stream_session_push_dev)
    int n_slots = 0, max_samples = 0, mask_words = 0;
    DevBuf slots, cache, mask, stage;  // stage: one push's entries, chunks and answers
    DevBuf dstate;                     // device pushes: SessDev arrays and the answers of sess_search
    SessDev D{};
    int32_t *dout = nullptr;
    void *pin = nullptr;               // pinned mirror of `stage`
    size_t pin_cap = 0;
    // host mirror per slot: samples cached, a read was started, last answer, settled; stamp: duplicate check of a push
    std::vector<int32_t> n, result, stamp;
    std::vector<uint8_t> live, settled;
    int32_t push_id = 0;
};

static int session_create(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots, int32_t max_samples, bool f32,
                          bool dev, adb_stream_session **out) {
    if (!ctx || !cfg || !out) { set_err("null argument"); return ADB_ERR_ARG; }
    *out = nullptr;
    if (n_slots < 1 || max_samples < 1) { set_err("n_slots and max_samples must be positive"); return ADB_ERR_ARG; }
    int rc = check_stream_config(cfg);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    adb_stream_session *s = new adb_stream_session();
    s->ctx = ctx;
    s->cfg = *cfg;
    s->f32 = f32;
    s->n_slots = n_slots;
    s->max_samples = max_samples;
    s->mask_words = (max_samples + 31) / 32;
    s->n.assign(n_slots, 0);
    s->result.assign(n_slots, 0);
    s->stamp.assign(n_slots, 0);
    s->live.assign(n_slots, 0);
    s->settled.assign(n_slots, 0);
    if (s->slots.ensure(sizeof(SessSlot) * (size_t)n_slots) || s->cache.ensure((f32 ? sizeof(float) : sizeof(int16_t)) * (size_t)n_slots * max_samples) ||
        s->mask.ensure(sizeof(uint32_t) * (size_t)n_slots * s->mask_words)) {
        adb_stream_session_destroy(s);
        set_err("cudaMalloc stream session arena");
        return ADB_ERR_CUDA;
    }
    if (cudaMemsetAsync(s->slots.p, 0, sizeof(SessSlot) * (size_t)n_slots, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        adb_stream_session_destroy(s);
        set_err("cudaMemset stream session state");
        return ADB_ERR_CUDA;
    }
    if (dev) {  // everything a device push needs, so that a push allocates nothing
        s->dev = true;
        const size_t ns = (size_t)n_slots;
        const size_t o_out = sizeof(SessEntry) * ns, o_err = o_out + sizeof(int32_t) * 2 * ns,
                     o_stamp = o_err + sizeof(unsigned long long), o_started = o_stamp + sizeof(uint32_t) * ns;
        if (s->dstate.ensure(o_started + ns)) {
            adb_stream_session_destroy(s);
            set_err("cudaMalloc stream session arena");
            return ADB_ERR_CUDA;
        }
        unsigned char *p = (unsigned char *)s->dstate.p;
        s->D.ent = (SessEntry *)p;
        s->dout = (int32_t *)(p + o_out);
        s->D.err = (unsigned long long *)(p + o_err);
        s->D.stamp = (uint32_t *)(p + o_stamp);
        s->D.started = p + o_started;
        s->D.n_slots = n_slots;
        if (cudaMemsetAsync(s->D.stamp, 0xff, sizeof(uint32_t) * ns, ctx->stream) != cudaSuccess ||
            cudaMemsetAsync(s->D.started, 0, ns, ctx->stream) != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
            adb_stream_session_destroy(s);
            set_err("cudaMemset stream session state");
            return ADB_ERR_CUDA;
        }
    }
    *out = s;
    return ADB_OK;
}

extern "C" int adb_stream_session_create(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots,
                                         int32_t max_samples, adb_stream_session **out) {
    return session_create(ctx, cfg, n_slots, max_samples, false, false, out);
}

extern "C" int adb_stream_session_create_f32(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots,
                                             int32_t max_samples, adb_stream_session **out) {
    return session_create(ctx, cfg, n_slots, max_samples, true, false, out);
}

extern "C" int adb_stream_session_create_dev(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots,
                                             int32_t max_samples, int32_t sig_type, adb_stream_session **out) {
    if (sig_type != ADB_SIG_I16 && sig_type != ADB_SIG_F32) {
        if (out) *out = nullptr;
        set_err("sig_type must be ADB_SIG_I16 or ADB_SIG_F32");
        return ADB_ERR_ARG;
    }
    return session_create(ctx, cfg, n_slots, max_samples, sig_type == ADB_SIG_F32, true, out);
}

extern "C" void adb_stream_session_destroy(adb_stream_session *s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    s->slots.release();
    s->cache.release();
    s->mask.release();
    s->stage.release();
    s->dstate.release();
    if (s->pin) cudaFreeHost(s->pin);
    delete s;
}

// true when no sample of src[0, n) is infinite or NaN (exponent bits all ones); copies them to dst unless it is null
static bool copy_finite(float *dst, const float *src, int64_t n) {
    uint32_t bad = 0;
    for (int64_t j = 0; j < n; j++) {
        uint32_t b;
        memcpy(&b, src + j, 4);
        if (dst) memcpy(dst + j, &b, 4);
        bad |= (b & 0x7f800000u) == 0x7f800000u;
    }
    return !bad;
}

// one push of either kind: `samples` is int16 ADC (with calibration on reset) or float32 pA, as the session holds
static int session_push(adb_stream_session *s, int32_t n, const int32_t *slots, const int64_t *chunk_offsets,
                        const void *samples, const uint8_t *reset, const float *calib_offset, const float *calib_scale,
                        int32_t *polya_start, uint8_t *settled) {
    const bool f32 = s->f32;
    const size_t esz = f32 ? sizeof(float) : sizeof(int16_t);
    if (n == 0) return ADB_OK;
    if (!slots || !chunk_offsets || !polya_start || !settled) { set_err("null argument"); return ADB_ERR_ARG; }
    if (chunk_offsets[0] < 0) { set_err("chunk_offsets must be non-negative"); return ADB_ERR_ARG; }
    for (int k = 0; k < n; k++)
        if (chunk_offsets[k + 1] < chunk_offsets[k]) { set_err("chunk_offsets must be non-decreasing"); return ADB_ERR_ARG; }
    if (chunk_offsets[n] > chunk_offsets[0] && !samples) {
        set_err(f32 ? "null pa with non-empty chunks" : "null adc with non-empty chunks");
        return ADB_ERR_ARG;
    }
    // validate the whole push before any state changes: a refused push leaves the session as it was
    if (++s->push_id == 0x7fffffff) { std::fill(s->stamp.begin(), s->stamp.end(), 0); s->push_id = 1; }
    for (int k = 0; k < n; k++) {
        const int sl = slots[k];
        if (sl < 0 || sl >= s->n_slots) { set_err("slot out of range"); return ADB_ERR_ARG; }
        if (s->stamp[sl] == s->push_id) { set_err("the same slot twice in one push"); return ADB_ERR_ARG; }
        s->stamp[sl] = s->push_id;
        if (reset && reset[k]) {
            if (f32) continue;  // float32 reads carry no calibration
            if (!calib_offset || !calib_scale) { set_err("a reset needs calib_offset and calib_scale"); return ADB_ERR_ARG; }
            if (!std::isfinite(calib_scale[k]) || !(calib_scale[k] > 0.f) || !std::isfinite(calib_offset[k])) {
                set_err("calibration scale must be finite and positive, offset finite");
                return ADB_ERR_ARG;
            }
        } else if (!s->live[sl]) {
            set_err("append to a slot that was never reset");
            return ADB_ERR_ARG;
        }
    }
    // entries that reach the device: resets and slots whose answer is not final; chunks are clipped at max_samples.
    // Float32 samples that do not reach the device (settled slot, beyond max_samples) are checked for finiteness here,
    // the others while they are staged.
    const float *pa = (const float *)samples;
    std::vector<SessEntry> ent;
    std::vector<int> ent_k;
    ent.reserve(n);
    int64_t total = 0;
    for (int k = 0; k < n; k++) {
        const int sl = slots[k];
        const bool rs = reset && reset[k];
        const int64_t clen = chunk_offsets[k + 1] - chunk_offsets[k];
        if (!rs && s->settled[sl]) {
            if (f32 && !copy_finite(nullptr, pa + chunk_offsets[k], clen)) { set_err("non-finite pA sample"); return ADB_ERR_ARG; }
            continue;
        }
        SessEntry E;
        E.slot = sl;
        E.reset = rs ? 1 : 0;
        const int64_t have = rs ? 0 : s->n[sl];
        E.len = (int32_t)std::min<int64_t>(clen, s->max_samples - have);
        E._pad = 0;
        E.src = total;
        E.coff = rs && !f32 ? calib_offset[k] : 0.f;
        E.cscale = rs && !f32 ? calib_scale[k] : 0.f;
        if (f32 && !copy_finite(nullptr, pa + chunk_offsets[k] + E.len, clen - E.len)) { set_err("non-finite pA sample"); return ADB_ERR_ARG; }
        total += E.len;
        ent.push_back(E);
        ent_k.push_back(k);
    }
    const int ne = (int)ent.size();
    if (ne > 0) {
        const size_t ent_bytes = (sizeof(SessEntry) * (size_t)ne + 15) & ~(size_t)15;
        const size_t blob_bytes = ((size_t)total * esz + 15) & ~(size_t)15;
        const size_t in_bytes = ent_bytes + blob_bytes, bytes = in_bytes + sizeof(int32_t) * 2 * (size_t)ne;
        CUDA_TRY(cudaSetDevice(s->ctx->device));
        if (bytes > s->pin_cap) {
            if (s->pin) cudaFreeHost(s->pin);
            s->pin = nullptr;
            s->pin_cap = 0;
            const size_t want = bytes + bytes / 4;
            CUDA_TRY(cudaHostAlloc(&s->pin, want, cudaHostAllocDefault));
            s->pin_cap = want;
        }
        if (s->stage.ensure(bytes)) { set_err("cudaMalloc stream session staging"); return ADB_ERR_CUDA; }
        unsigned char *hp = (unsigned char *)s->pin;
        memcpy(hp, ent.data(), sizeof(SessEntry) * (size_t)ne);
        unsigned char *hb = hp + ent_bytes;
        for (int q = 0; q < ne; q++) {
            if (ent[q].len <= 0) continue;
            const int64_t o = chunk_offsets[ent_k[q]];
            if (!f32) {
                memcpy((int16_t *)hb + ent[q].src, (const int16_t *)samples + o, sizeof(int16_t) * (size_t)ent[q].len);
            } else if (!copy_finite((float *)hb + ent[q].src, pa + o, ent[q].len)) {
                set_err("non-finite pA sample");
                return ADB_ERR_ARG;
            }
        }
        cudaStream_t st = s->ctx->stream;
        CUDA_TRY(cudaMemcpyAsync(s->stage.p, hp, in_bytes, cudaMemcpyHostToDevice, st));
        unsigned char *dp = (unsigned char *)s->stage.p;
        const int ablocks = (ne + SESS_APPEND_WARPS - 1) / SESS_APPEND_WARPS;
        if (!f32) {
            SessArgs A;
            A.slots = (SessSlot *)s->slots.p;
            A.cache = (int16_t *)s->cache.p;
            A.mask = (uint32_t *)s->mask.p;
            A.ent = (const SessEntry *)dp;
            A.blob = (const int16_t *)(dp + ent_bytes);
            A.out = (int32_t *)(dp + in_bytes);
            A.n_ent = ne;
            A.max_samples = s->max_samples;
            A.mask_words = s->mask_words;
            stream_append_kernel<<<ablocks, SESS_APPEND_WARPS * 32, 0, st>>>(A, s->cfg);
            CUDA_TRY(cudaGetLastError());
            stream_search_kernel<<<ne, ADB_VAL_THREADS, 0, st>>>(A, s->cfg);
        } else {
            SessArgsF32 A;
            A.slots = (SessSlot *)s->slots.p;
            A.cache = (float *)s->cache.p;
            A.mask = (uint32_t *)s->mask.p;
            A.ent = (const SessEntry *)dp;
            A.blob = (const float *)(dp + ent_bytes);
            A.out = (int32_t *)(dp + in_bytes);
            A.n_ent = ne;
            A.max_samples = s->max_samples;
            A.mask_words = s->mask_words;
            stream_append_f32_kernel<<<ablocks, SESS_APPEND_WARPS * 32, 0, st>>>(A, s->cfg);
            CUDA_TRY(cudaGetLastError());
            stream_search_f32_kernel<<<ne, ADB_VAL_THREADS, 0, st>>>(A, s->cfg);
        }
        CUDA_TRY(cudaGetLastError());
        s->ctx->launches += 2;
        CUDA_TRY(cudaMemcpyAsync(hp + in_bytes, dp + in_bytes, sizeof(int32_t) * 2 * (size_t)ne, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        const int32_t *res = (const int32_t *)(hp + in_bytes);
        for (int q = 0; q < ne; q++) {
            const int sl = ent[q].slot;
            s->n[sl] = (ent[q].reset ? 0 : s->n[sl]) + ent[q].len;
            s->live[sl] = 1;
            s->result[sl] = res[2 * q];
            s->settled[sl] = res[2 * q + 1] ? 1 : 0;
        }
    }
    for (int k = 0; k < n; k++) {
        polya_start[k] = s->result[slots[k]];
        settled[k] = s->settled[slots[k]];
    }
    return ADB_OK;
}

extern "C" int adb_stream_session_push(adb_stream_session *s, int32_t n, const int32_t *slots, const int64_t *chunk_offsets,
                                       const int16_t *adc, const uint8_t *reset, const float *calib_offset,
                                       const float *calib_scale, int32_t *polya_start, uint8_t *settled) {
    if (!s || n < 0) { set_err("invalid argument"); return ADB_ERR_ARG; }
    if (s->dev) { set_err("host push on a device-push session"); return ADB_ERR_ARG; }
    if (s->f32) { set_err("int16 push on a float32 session"); return ADB_ERR_ARG; }
    return session_push(s, n, slots, chunk_offsets, adc, reset, calib_offset, calib_scale, polya_start, settled);
}

extern "C" int adb_stream_session_push_f32(adb_stream_session *s, int32_t n, const int32_t *slots,
                                           const int64_t *chunk_offsets, const float *pa, const uint8_t *reset,
                                           int32_t *polya_start, uint8_t *settled) {
    if (!s || n < 0) { set_err("invalid argument"); return ADB_ERR_ARG; }
    if (s->dev) { set_err("host push on a device-push session"); return ADB_ERR_ARG; }
    if (!s->f32) { set_err("float32 push on an int16 session"); return ADB_ERR_ARG; }
    return session_push(s, n, slots, chunk_offsets, pa, reset, nullptr, nullptr, polya_start, settled);
}

// the adb_last_error() text of each refusal of session_push, by SessReason
static const char *const kSessReasonText[SESS_R_COUNT] = {
    nullptr,
    "chunk_offsets must be non-negative",
    "chunk_offsets must be non-decreasing",
    "null adc with non-empty chunks",
    "null pa with non-empty chunks",
    "slot out of range",
    "the same slot twice in one push",
    "a reset needs calib_offset and calib_scale",
    "calibration scale must be finite and positive, offset finite",
    "append to a slot that was never reset",
    "non-finite pA sample",
};

extern "C" const char *adb_stream_session_reason(int32_t reason) {
    return reason > SESS_R_NONE && reason < SESS_R_COUNT ? kSessReasonText[reason] : nullptr;
}

extern "C" int adb_stream_session_push_dev(adb_stream_session *s, int32_t n, const int32_t *slots,
                                           const int64_t *chunk_offsets, const void *samples, const uint8_t *reset,
                                           const float *calib_offset, const float *calib_scale, int32_t *polya_start,
                                           uint8_t *settled, int32_t *status, void *cuda_stream) {
    if (!s || n < 0) { set_err("invalid argument"); return ADB_ERR_ARG; }
    if (!s->dev) { set_err("device push on a host-push session"); return ADB_ERR_ARG; }
    if (n > s->n_slots) { set_err("more entries than slots: a push names each slot at most once"); return ADB_ERR_ARG; }
    if (!status || !chunk_offsets || (n > 0 && (!slots || !polya_start || !settled))) { set_err("null argument"); return ADB_ERR_ARG; }
    if (s->f32 && (calib_offset || calib_scale)) { set_err("a float32 session takes no calibration"); return ADB_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(s->ctx->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (n == 0) {
        CUDA_TRY(cudaMemsetAsync(status, 0, sizeof(int32_t) * 2, st));
        return ADB_OK;
    }
    SessPush Q;
    Q.slots = slots;
    Q.offs = chunk_offsets;
    Q.samples = samples;
    Q.reset = reset;
    Q.coff = calib_offset;
    Q.cscale = calib_scale;
    Q.polya_start = polya_start;
    Q.settled = settled;
    Q.status = status;
    Q.n = n;
    const int eblocks = (n + SESS_DEV_THREADS - 1) / SESS_DEV_THREADS;
    // float32: enough CTAs for the finiteness scan, whose length only the device knows
    const int cblocks = s->f32 ? std::max(eblocks, 4 * s->ctx->sm_count) : eblocks;
    const int ablocks = (n + SESS_APPEND_WARPS - 1) / SESS_APPEND_WARPS;
    stream_dev_stamp_kernel<<<eblocks, SESS_DEV_THREADS, 0, st>>>(Q, s->D);
    CUDA_TRY(cudaGetLastError());
    if (!s->f32) {
        SessArgs A;
        A.slots = (SessSlot *)s->slots.p;
        A.cache = (int16_t *)s->cache.p;
        A.mask = (uint32_t *)s->mask.p;
        A.ent = s->D.ent;
        A.blob = (const int16_t *)samples;
        A.out = s->dout;
        A.n_ent = n;
        A.max_samples = s->max_samples;
        A.mask_words = s->mask_words;
        stream_dev_check_kernel<<<cblocks, SESS_DEV_THREADS, 0, st>>>(A, Q, s->D);
        CUDA_TRY(cudaGetLastError());
        stream_append_dev_kernel<<<ablocks, SESS_APPEND_WARPS * 32, 0, st>>>(A, s->cfg, s->D);
        CUDA_TRY(cudaGetLastError());
        stream_search_dev_kernel<<<n, ADB_VAL_THREADS, 0, st>>>(A, s->cfg, s->D, Q);
    } else {
        SessArgsF32 A;
        A.slots = (SessSlot *)s->slots.p;
        A.cache = (float *)s->cache.p;
        A.mask = (uint32_t *)s->mask.p;
        A.ent = s->D.ent;
        A.blob = (const float *)samples;
        A.out = s->dout;
        A.n_ent = n;
        A.max_samples = s->max_samples;
        A.mask_words = s->mask_words;
        stream_dev_check_f32_kernel<<<cblocks, SESS_DEV_THREADS, 0, st>>>(A, Q, s->D);
        CUDA_TRY(cudaGetLastError());
        stream_append_dev_f32_kernel<<<ablocks, SESS_APPEND_WARPS * 32, 0, st>>>(A, s->cfg, s->D);
        CUDA_TRY(cudaGetLastError());
        stream_search_dev_f32_kernel<<<n, ADB_VAL_THREADS, 0, st>>>(A, s->cfg, s->D, Q);
    }
    CUDA_TRY(cudaGetLastError());
    s->ctx->launches += 4;
    return ADB_OK;
}

// ---- CNN scores (kernel-level test entry) ------------------------------------------------------------------------
extern "C" int adb_cnn_scores_host(adb_ctx *ctx, const float *x, int32_t n, int32_t L, const float *cnn_weights, float *scores) {
    if (!ctx || !x || !cnn_weights || !scores || n < 0 || L < CNN_K) { set_err("invalid argument"); return ADB_ERR_ARG; }
    if (n == 0) return ADB_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CnnDims D;
    D.Lx = L;
    D.L1 = (L + 2 * 3 - CNN_K) / 3 + 1;
    D.LP = (D.L1 + 3) & ~3;
    D.Lout = (D.L1 - 1) * 3 - 2 * 3 + CNN_K;
    if (ctx->cnn_x.ensure(sizeof(float) * (size_t)n * L) || ctx->cnn_scores.ensure(sizeof(float) * (size_t)n * 2 * D.Lout) ||
        ctx->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc cnn buffers"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(ctx->cnn_x.p, x, sizeof(float) * (size_t)n * L, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, st));
    int rc = cnn_forward_dev(ctx, (const float *)ctx->cnn_x.p, n, D, (const float *)ctx->h_misc2.p, (float *)ctx->cnn_scores.p, st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(scores, ctx->cnn_scores.p, sizeof(float) * (size_t)n * 2 * D.Lout, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- c_llr_trace ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) llr_trace_kernel(const double *signals, const int64_t *offs, const int64_t *params,
                                                        double *gains, double *c_out, double *c2_out, double *c_tmp,
                                                        double *c2_tmp) {
    __shared__ int tmp[2];
    const int t = blockIdx.x;
    const int64_t o = offs[t];
    const int n = (int)(offs[t + 1] - o);
    const int64_t *p = params + (size_t)t * 11;
    const int start = (int)p[0], end = (int)p[1], head = (int)p[2], tail = (int)p[3], stride = (int)max((int64_t)1, p[4]);
    const int aes = (int)p[5], aw = (int)p[6], as_ = (int)p[7], pes = (int)p[8], pw = (int)p[9], ps = (int)p[10];
    const double *x = signals + o;
    double *c = (c_out ? c_out : c_tmp) + o, *c2 = (c2_out ? c2_out : c2_tmp) + o, *g = gains + o;
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < n; i++) { s = __dadd_rn(s, x[i]); c[i] = s; }
    } else if (threadIdx.x == 32) {
        double s2 = 0.0;
        for (int i = 0; i < n; i++) { s2 = __dadd_rn(s2, __dmul_rn(x[i], x[i])); c2[i] = s2; }
    }
    __threadfence_block();
    __syncthreads();
    if (n <= 0 || end > n || start < 0 || end < 1) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) g[i] = 0.0;
        return;
    }
    cta_llr_gains(c, c2, n, start, end, head, tail, stride, g);
    const int mode = pes > 0 ? 2 : (aes > 0 ? 1 : 0);
    if (mode) cta_llr_early_stop(g, n, start, end, head, tail, stride, mode, aw, max(as_, 1), pw, max(ps, 1), tmp);
}

extern "C" int adb_llr_trace_host(adb_ctx *ctx, const double *signals, const int64_t *sig_offsets, int32_t n_traces,
                                  const int64_t *params, double *gains, double *c, double *c2) {
    if (!ctx || !signals || !sig_offsets || !params || !gains || n_traces < 0) { set_err("null argument"); return ADB_ERR_ARG; }
    if (n_traces == 0) return ADB_OK;
    for (int t = 0; t < n_traces; t++) {
        const int64_t *p = params + (size_t)t * 11;
        const int64_t stride = std::max<int64_t>(1, p[4]);
        if ((p[8] > 0 || p[5] > 0) && (p[7] <= 0 || p[7] % stride != 0)) { set_err("early_stop_stride % stride != 0"); return ADB_ERR_ARG; }
        if (p[8] > 0 && (p[10] <= 0 || p[10] % stride != 0)) { set_err("polya early_stop_stride % stride != 0"); return ADB_ERR_ARG; }
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t total = (size_t)sig_offsets[n_traces];
    DevBuf &dx = ctx->h_signal, &dg = ctx->h_records, &dc = ctx->h_misc2, &dc2 = ctx->h_misc3, &doff = ctx->h_offsets, &dp = ctx->h_misc;
    if (dx.ensure(total * 8 + 8) || dg.ensure(total * 8 + 8) || dc.ensure(total * 8 + 8) || dc2.ensure(total * 8 + 8) ||
        doff.ensure(sizeof(int64_t) * ((size_t)n_traces + 1)) || dp.ensure(sizeof(int64_t) * 11 * (size_t)n_traces)) {
        set_err("cudaMalloc llr trace buffers");
        return ADB_ERR_CUDA;
    }
    CUDA_TRY(cudaMemcpyAsync(dx.p, signals, total * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(doff.p, sig_offsets, sizeof(int64_t) * ((size_t)n_traces + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dp.p, params, sizeof(int64_t) * 11 * (size_t)n_traces, cudaMemcpyHostToDevice, st));
    llr_trace_kernel<<<n_traces, 128, 0, st>>>((const double *)dx.p, (const int64_t *)doff.p, (const int64_t *)dp.p,
                                               (double *)dg.p, nullptr, nullptr, (double *)dc.p, (double *)dc2.p);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(gains, dg.p, total * 8, cudaMemcpyDeviceToHost, st));
    if (c) CUDA_TRY(cudaMemcpyAsync(c, dc.p, total * 8, cudaMemcpyDeviceToHost, st));
    if (c2) CUDA_TRY(cudaMemcpyAsync(c2, dc2.p, total * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- peak picking (kernel-level test entry) -----------------------------------------------------------------------------
#define ADB_PEAKS_MAX_N 4096
__global__ void __launch_bounds__(ADB_TRACE_THREADS) peaks_test_kernel(const double *traces, const int64_t *offs, const double *params,
                                                                    int nds_max, int peak_cap, int *out) {
    extern __shared__ __align__(16) unsigned char smem[];
    const TraceScratch T = trace_scratch_from(smem, nds_max, peak_cap);
    const int t = blockIdx.x;
    const int n = (int)(offs[t + 1] - offs[t]);
    const double *p = params + (size_t)t * 8;
    const int mode = (int)p[0], dist = (int)p[1], want = min(max((int)p[5], 0), 32), n2n = (int)p[6];
    const double pmin = p[2], wmin = p[3], rel_height = p[4];
    int *res = out + (size_t)t * 33;
    double *g = T.trace;
    for (int i = threadIdx.x; i < n; i += blockDim.x) g[i] = traces[offs[t] + i];
    __syncthreads();
    if (mode == 0) {
        TraceView W;
        W.x = g; W.n = n; W.nan2num = n2n;
        const int npk = cta_peaks_prepare(W, pmin, wmin, rel_height, T.PS, T.itmp);
        if (threadIdx.x < 32) {
            int pk[32];
            const int k = warp_peaks_select(W, npk, dist, pmin, wmin, rel_height, want, pk, T.PS);
            if (threadIdx.x == 0) {
                res[0] = k;
                for (int i = 0; i < k; i++) res[1 + i] = pk[i];
            }
        }
    } else if (mode == 1) {
        int s0, e0;
        cta_trace_support(g, n, s0, e0, T.itmp);
        if (threadIdx.x < 32) { const double sd = warp_nanstd(g, s0, e0); if (threadIdx.x == 0) T.dtmp[0] = sd; }
        __syncthreads();
        const int ae = cta_adapter_end(g, n, s0, e0, __dmul_rn(pmin, T.dtmp[0]), wmin, rel_height, T.PS, T.itmp + 4);
        if (threadIdx.x == 0) { res[0] = 1; res[1] = ae; }
    } else {
        const int pe = cta_polya_end(g, n, T.PS, T.itmp + 4);
        if (threadIdx.x == 0) { res[0] = 1; res[1] = pe; }
    }
}

extern "C" int adb_find_peaks_host(adb_ctx *ctx, const double *traces, const int64_t *offsets, int32_t n_traces,
                                   const double *params, int32_t *out) {
    if (!ctx || !traces || !offsets || !params || !out || n_traces < 0) { set_err("null argument"); return ADB_ERR_ARG; }
    if (n_traces == 0) return ADB_OK;
    int n_max = 0;
    for (int t = 0; t < n_traces; t++) {
        const int64_t n = offsets[t + 1] - offsets[t];
        if (n < 0 || n > ADB_PEAKS_MAX_N) { set_err("trace length outside [0, 4096]"); return ADB_ERR_ARG; }
        n_max = std::max(n_max, (int)n);
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t total = (size_t)offsets[n_traces];
    DevBuf &dx = ctx->h_signal, &doff = ctx->h_offsets, &dp = ctx->h_misc, &dout = ctx->h_records;
    if (dx.ensure(total * 8 + 8) || doff.ensure(sizeof(int64_t) * ((size_t)n_traces + 1)) || dp.ensure(sizeof(double) * 8 * (size_t)n_traces) ||
        dout.ensure(sizeof(int) * 33 * (size_t)n_traces)) { set_err("cudaMalloc peak test buffers"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(dx.p, traces, total * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(doff.p, offsets, sizeof(int64_t) * ((size_t)n_traces + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dp.p, params, sizeof(double) * 8 * (size_t)n_traces, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(dout.p, 0, sizeof(int) * 33 * (size_t)n_traces, st));
    const int nds_max = std::max(64, n_max + 2), peak_cap = nds_max / 2 + 24;
    const size_t smem = trace_smem_bytes(nds_max, peak_cap);
    if ((int)smem > ctx->max_smem_optin) { set_err("trace does not fit in shared memory"); return ADB_ERR_UNSUPPORTED; }
    CUDA_TRY(cudaFuncSetAttribute(peaks_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    peaks_test_kernel<<<n_traces, ADB_TRACE_THREADS, smem, st>>>((const double *)dx.p, (const int64_t *)doff.p, (const double *)dp.p,
                                                                 nds_max, peak_cap, (int *)dout.p);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, dout.p, sizeof(int) * 33 * (size_t)n_traces, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- legacy three-split detectors -----------------------------------------------------------------------------------
extern "C" int adb_llr_detect_host(adb_ctx *ctx, const double *signals, const int64_t *sig_offsets, int32_t n_signals,
                                   const int64_t *params, int64_t *out) {
    if (!ctx || !signals || !sig_offsets || !params || !out || n_signals < 0) { set_err("null argument"); return ADB_ERR_ARG; }
    if (n_signals == 0) return ADB_OK;
    for (int t = 0; t < n_signals; t++)
        if (params[3 * (size_t)t] < 0 || params[3 * (size_t)t + 1] < 0) { set_err("negative min_obs_adapter / border_trim"); return ADB_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t total = (size_t)sig_offsets[n_signals];
    DevBuf &dx = ctx->h_signal, &dc = ctx->h_misc2, &dc2 = ctx->h_misc3, &doff = ctx->h_offsets, &dp = ctx->h_misc, &dout = ctx->h_records;
    if (dx.ensure(total * 8 + 8) || dc.ensure(total * 8 + 8) || dc2.ensure(total * 8 + 8) ||
        doff.ensure(sizeof(int64_t) * ((size_t)n_signals + 1)) || dp.ensure(sizeof(int64_t) * 3 * (size_t)n_signals) ||
        dout.ensure(sizeof(int64_t) * 4 * (size_t)n_signals)) {
        set_err("cudaMalloc llr detect buffers");
        return ADB_ERR_CUDA;
    }
    CUDA_TRY(cudaMemcpyAsync(dx.p, signals, total * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(doff.p, sig_offsets, sizeof(int64_t) * ((size_t)n_signals + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dp.p, params, sizeof(int64_t) * 3 * (size_t)n_signals, cudaMemcpyHostToDevice, st));
    llr_legacy_detect_kernel<<<n_signals, ADB_LEGACY_THREADS, 0, st>>>((const double *)dx.p, (const int64_t *)doff.p,
                                                                       (const int64_t *)dp.p, (double *)dc.p, (double *)dc2.p,
                                                                       (int64_t *)dout.p);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, dout.p, sizeof(int64_t) * 4 * (size_t)n_signals, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- downscale ------------------------------------------------------------------------------------------------------
__global__ void downscale_kernel(BatchDev B, int col0, int factor, int ncols_out, float *out) {
    const int r = blockIdx.y;
    const ReadSrc src = make_src(B, r);
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < ncols_out; b += gridDim.x * blockDim.x) {
        const int j0 = col0 + b * factor;
        bool nan = false;
        for (int k = 0; k < factor; k++) { int j = j0 + k; if (j < B.m && j >= src.n) nan = true; }
        float v;
        if (nan) v = CUDART_NAN_F;
        else v = block_mean_f32([&](int k) { int j = j0 + k; return (j < B.m) ? src.pa(j) : 0.0f; }, factor);
        out[(size_t)r * ncols_out + b] = v;
    }
}

extern "C" int adb_downscale_host(adb_ctx *ctx, const adb_batch *batch, int32_t col0, int32_t factor, float *out) {
    if (!ctx || !out || factor < 1 || factor > 128 || col0 < 0) { set_err("invalid argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StagedBatch sb;
    rc = stage_batch(ctx, batch, &sb, st);
    if (rc) return rc;
    const int ncols = (std::max(batch->m - col0, 0) + factor - 1) / factor;
    if (ncols == 0 || batch->n_reads == 0) return ADB_OK;
    if (ctx->h_records.ensure(sizeof(float) * (size_t)ncols * batch->n_reads)) { set_err("cudaMalloc downscale"); return ADB_ERR_CUDA; }
    dim3 grid((ncols + 127) / 128, batch->n_reads);
    downscale_kernel<<<grid, 128, 0, st>>>(to_dev_view(sb.dev), col0, factor, ncols, (float *)ctx->h_records.p);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, ctx->h_records.p, sizeof(float) * (size_t)ncols * batch->n_reads, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

// ---- full open-pore lists (reads whose list overflows the record) ---------------------------------------------------
#include "adb_openpore.cuh"

extern "C" int adb_open_pores_host(adb_ctx *ctx, const adb_batch *batch, const int32_t *sel, int32_t n_sel,
                                   const int32_t *seg_begin, const int32_t *seg_end, int64_t *out_offsets,
                                   int32_t *out_pos, int64_t cap) {
    if (!ctx || !sel || !seg_begin || !seg_end || !out_offsets || n_sel < 0 || cap < 0 || (cap > 0 && !out_pos)) {
        set_err("invalid argument");
        return ADB_ERR_ARG;
    }
    int rc = check_batch(batch);
    if (rc) return rc;
    out_offsets[0] = 0;
    if (n_sel == 0) return ADB_OK;
    // compact sub-batch of the selected reads (host side gather: the call is rare and touches a few reads)
    std::vector<int64_t> offs((size_t)n_sel + 1, 0);
    std::vector<int32_t> lens(n_sel), seg((size_t)n_sel * 2);
    std::vector<float> coff(n_sel), cscale(n_sel);
    std::vector<unsigned char> blob;
    const size_t esz = batch->sig_type == ADB_SIG_F32 ? 4 : 2;
    for (int k = 0; k < n_sel; k++) {
        const int r = sel[k];
        if (r < 0 || r >= batch->n_reads) { set_err("selection outside the batch"); return ADB_ERR_ARG; }
        int64_t o0, n;
        if (batch->sig_type == ADB_SIG_F32) { o0 = (int64_t)r * batch->m; n = batch->m; }
        else {
            o0 = batch->offsets[r];
            n = std::min<int64_t>(batch->offsets[r + 1] - o0, batch->m);
            coff[k] = batch->calib_offset[r];
            cscale[k] = batch->calib_scale[r];
        }
        lens[k] = batch->full_lens[r];
        seg[2 * k] = seg_begin[k];
        seg[2 * k + 1] = seg_end[k];
        const unsigned char *src = (const unsigned char *)batch->signal + (size_t)o0 * esz;
        blob.insert(blob.end(), src, src + (size_t)n * esz);
        offs[k + 1] = offs[k] + n;
    }
    adb_batch sub = *batch;
    sub.signal = blob.data();
    sub.n_reads = n_sel;
    sub.batch_size = n_sel;
    sub.full_lens = lens.data();
    if (batch->sig_type == ADB_SIG_I16) { sub.offsets = offs.data(); sub.calib_offset = coff.data(); sub.calib_scale = cscale.data(); }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StagedBatch sb;
    rc = stage_batch(ctx, &sub, &sb, st);
    if (rc) return rc;
    const size_t nb_seg = sizeof(int) * 2 * (size_t)n_sel, nb_cnt = sizeof(long long) * ((size_t)n_sel + 1);
    if (ctx->h_misc.ensure(nb_seg + 2 * nb_cnt + 64)) { set_err("cudaMalloc open-pore scratch"); return ADB_ERR_CUDA; }
    int *d_seg = (int *)ctx->h_misc.p;
    long long *d_cnt = (long long *)((unsigned char *)ctx->h_misc.p + ((nb_seg + 15) & ~(size_t)15));
    long long *d_off = d_cnt + n_sel + 1;
    CUDA_TRY(cudaMemcpyAsync(d_seg, seg.data(), nb_seg, cudaMemcpyHostToDevice, st));
    OpenPoreArgs A;
    A.B = to_dev_view(sb.dev);
    A.seg = d_seg;
    A.counts = d_cnt;
    A.offs = nullptr;
    A.out = nullptr;
    A.cap = 0;
    open_pores_full_kernel<<<n_sel, ADB_OP_THREADS, 0, st>>>(A);
    std::vector<long long> cnt(n_sel);
    CUDA_TRY(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(long long) * (size_t)n_sel, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    std::vector<long long> off((size_t)n_sel + 1, 0);
    for (int k = 0; k < n_sel; k++) { off[k + 1] = off[k] + cnt[k]; out_offsets[k + 1] = off[k + 1]; }
    ctx->launches += 1;
    const long long total = off[n_sel];
    if (total == 0 || cap < total) return ADB_OK;  // cap too small: the caller sizes the buffer from out_offsets[n_sel]
    if (ctx->h_records.ensure(sizeof(int) * (size_t)total)) { set_err("cudaMalloc open-pore output"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(d_off, off.data(), sizeof(long long) * ((size_t)n_sel + 1), cudaMemcpyHostToDevice, st));
    A.counts = nullptr;
    A.offs = d_off;
    A.out = (int *)ctx->h_records.p;
    A.cap = total;
    open_pores_full_kernel<<<n_sel, ADB_OP_THREADS, 0, st>>>(A);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_pos, A.out, sizeof(int) * (size_t)total, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ADB_OK;
}

#include "adb_ingest.cuh"
#include "adb_files.cuh"


#ifdef ADB_VH_STATS
// instrumented builds only (tools/vhstats.py): per-phase cycle counters of validate_hist_kernel; reset != 0 clears them
extern "C" int adb_vh_stats(unsigned long long *out, int reset) {
    if (cudaMemcpyFromSymbol(out, vh_dbg, sizeof(unsigned long long) * 16) != cudaSuccess) return ADB_ERR_CUDA;
    if (reset) { unsigned long long z[16] = {0}; if (cudaMemcpyToSymbol(vh_dbg, z, sizeof(z)) != cudaSuccess) return ADB_ERR_CUDA; }
    return ADB_OK;
}
#endif
