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

// adb_ctx_set_option switches; the pipelined entry points copy them onto the twin in one assignment
struct AdbOptions {
    int copy_only = 0;           // "pipeline_copy_only": pipelined entry points skip the kernels
    int no_fast_validate = 0;    // "no_fast_validate"
    int hist_validate = 1;       // "hist_validate" 0: counting passes (validate_fast_kernel) instead of the tensor-core histograms (adb_vhist.cuh)
    int no_cand_followup = 0;    // "no_cand_followup": further poly(A) candidates go to validate_kernel (A/B)
    int cnn_fp32 = 0;            // "cnn_fp32_pipe": 64->64 convolutions on the FP32 pipe instead of tcgen05
    int cnn_tc_per_read = 0;     // "cnn_tc_per_read_tiles": tensor-core convolution tiles restart at every read instead of walking the packed row stream (A/B)
    int exact_gsel = 0;          // "exact_global_select": always use the multi-pass select
    int host_zstd = 0;           // "host_zstd": adb_detect_files decompresses zstd frames on the host (A/B)
};

// device staging of one chunk of the pipelined entry points (adb_ingest.cuh)
struct ChunkBufs {
    DevBuf signal, offsets, lens, coff, cscale, records, status;
    DevBuf comp, coffs, nsamp;  // svb16 streams, their offsets, samples per read
    DevBuf frames, foffs, zstat;  // zstd frames, their offsets, per-frame status
    cudaEvent_t copied = nullptr, done = nullptr;  // the chunk's H2D copies / its D2H copies have finished
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
    AdbOptions opt;
    ChunkBufs p[2];  // double-buffered staging for the pipelined entry points
    DevBuf z_fail;   // VBZ ingest: frames the device refused
    // pinned slot ring of adb_detect_files, kept between calls (pinning gigabytes costs seconds)
    void *file_ring = nullptr;
    void (*file_ring_free)(void *) = nullptr;
    // scratch (device)
    DevBuf states, hist, series, given, status;
    DevBuf gsb_plan, gsb_hist, gsb_tab, gsb_bases, gsb_active;  // sampled one-pass global select
    DevBuf mvs_perm;           // length-sorted read order of mvs_series_kernel
    DevBuf llr_cc;             // prefix sums of llr_primary_kernel (per resident CTA)
    DevBuf vf_done;            // per-read flags of validate_fast_kernel
    int ct_slot = -1;          // this context's slot of the constant bank adb_c_convT (adb_cnn_tc.cuh), -1: none left
    int cnn_a0t_geom[3] = {-1, -1, -1};  // (L1, rows per read, rows per octet) the tile-layout activation buffer was last zeroed for
    int vf_last_reads = 0;
    int gsb_last_batches = 0;
    int64_t zstd_host_frames = 0;  // adb_ctx_query("zstd_host_frames"): frames the last call decompressed on the host
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

