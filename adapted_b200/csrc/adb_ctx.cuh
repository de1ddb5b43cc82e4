// Host-side context shared by the entry points (not part of the ABI: adb_ctx is opaque to callers).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <utility>
#include <vector>

#include "../../include/adapted_b200.h"

inline std::string &adb_err_string() {
    static thread_local std::string s;
    return s;
}
inline void set_err(const std::string &s) { adb_err_string() = s; }

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_err(std::string(#expr) + ": " + cudaGetErrorString(_e));                       \
            return ADB_ERR_CUDA;                                                               \
        }                                                                                      \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4;
        if (cudaMalloc(&p, want) != cudaSuccess) {
            if (cudaMalloc(&p, bytes) != cudaSuccess) return -1;
            want = bytes;
        }
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct adb_ctx {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    int64_t launches = 0;
    // second context of the pipelined ingest: consecutive chunks alternate between the two (own stream, own scratch), so
    // the thin tail of one chunk (moving statistics of its longest reads, handed-over reads) runs under the wide head
    // of the next
    adb_ctx *twin = nullptr;
    // optional per-kernel-class timing (bench.py roofline): events bracket every launch of a class
    int timing = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[8];  // see ADB_TC_* in adb_api.cu
    double timing_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int64_t timing_n[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // double-buffered staging for the pipelined host entry point
    DevBuf p_signal[2], p_offsets[2], p_lens[2], p_coff[2], p_cscale[2], p_records[2], p_status[2];
    DevBuf p_comp[2], p_coffs[2], p_nsamp[2];  // compressed ingest: svb16 streams, their offsets, samples per read
    DevBuf p_frames[2], p_foffs[2], p_zstat[2];  // VBZ ingest: zstd frames, their offsets, per-frame status
    DevBuf z_fail;                                 // VBZ ingest: frames the device refused (one counter per call)
    int opt_copy_only = 0;     // adb_ctx_set_option("pipeline_copy_only"): pipelined entry points skip the kernels
    // pinned slot ring of adb_detect_files, kept between calls (pinning gigabytes costs seconds)
    void *file_ring = nullptr;
    void (*file_ring_free)(void *) = nullptr;
    cudaEvent_t p_done[2] = {nullptr, nullptr}, p_copied[2] = {nullptr, nullptr};
    // scratch (device)
    DevBuf states, hist, series, given, status;
    DevBuf gsb_plan, gsb_hist, gsb_tab, gsb_bases, gsb_active;  // sampled one-pass global select
    DevBuf mvs_perm;           // length-sorted read order of mvs_series_kernel
    DevBuf llr_cc;             // prefix sums of llr_primary_kernel (per resident CTA)
    DevBuf vf_done;            // per-read flags of validate_fast_kernel
    int ct_slot = -1;          // this context's slot of the constant bank adb_c_convT (adb_cnn_tc.cuh), -1: none left
    int opt_no_fast_validate = 0;
    int opt_hist_validate = 1;  // adb_ctx_set_option("hist_validate", 0): counting passes (validate_fast_kernel) instead of the tensor-core histograms (adb_vhist.cuh)
    int opt_no_cand_followup = 0;  // adb_ctx_set_option("no_cand_followup"): further poly(A) candidates go to validate_kernel (A/B)
    int cnn_a0t_l1 = -1;       // L1 the tile-layout activation buffer was last zeroed for
    int opt_cnn_fp32 = 0;      // adb_ctx_set_option("cnn_fp32_pipe"): 64->64 convolutions on the FP32 pipe instead of tcgen05
    int vf_last_reads = 0;
    int gsb_last_batches = 0;
    int opt_exact_gsel = 0;
    int opt_host_zstd = 0;        // adb_ctx_set_option("host_zstd"): adb_detect_files decompresses zstd frames on the host (A/B)
    int64_t zstd_host_frames = 0;  // adb_ctx_query("zstd_host_frames"): frames the last call decompressed on the host  // adb_ctx_set_option("exact_global_select"): always use the multi-pass select
    DevBuf cnn_x, cnn_act0, cnn_act1, cnn_scores, cnn_w, cnn_aux, cnn_post, sp_rows, cnn_wtc, cnn_a0t, cnn_ct;
    DevBuf val_cc;  // hail-mary prefix sums of the unstaged validate_kernel: [grid][2][nds_max] doubles
    // staging for the *_host entry points
    DevBuf h_signal, h_offsets, h_lens, h_coff, h_cscale, h_records, h_misc, h_misc2, h_misc3;
};

struct KernelTimer {  // brackets one launch with events when ctx->timing is on
    adb_ctx *ctx;
    int cls;
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    KernelTimer(adb_ctx *c, int cls_, cudaStream_t s) : ctx(c), cls(cls_), st(s) {
        if (ctx->timing) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, st);
        }
    }
    ~KernelTimer() {
        if (ctx->timing) {
            cudaEventRecord(b, st);
            ctx->ev[cls].push_back({a, b});
        }
    }
};

