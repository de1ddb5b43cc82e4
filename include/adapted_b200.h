/*
 * adapted_b200 -- C ABI of the B200-native boundary-detection hot path (drop-in for KleistLab/ADAPTed v0.2.4).
 *
 * The reference has no FFI of its own (it is python + one Cython module); the entry points below are what a
 * binding for the hot path replaces.  Each one cites the reference interface it stands in for
 * (paths relative to the reference repository).  INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *   - plain C, pointers + sizes, no torch / C++ types;
 *   - every function returns 0 on success or a negative adb_status; adb_last_error() gives the text;
 *   - "_host" variants take HOST buffers (pageable or pinned), do H2D / D2H themselves and are synchronous;
 *   - "_dev" variants take DEVICE pointers and a cudaStream_t (as void*), and are asynchronous on that stream;
 *   - all kernels are hand-written sm_100a CUDA; there is NO CPU fallback: without a CUDA device every compute
 *     entry point fails with ADB_ERR_CUDA.
 */
#ifndef ADAPTED_B200_H
#define ADAPTED_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADB_ABI_VERSION 1
#define ADB_MAX_CAND 16        /* >= cnn_boundaries.polya_cand_k (10 / 15 in the shipped configs)            */
#define ADB_MAX_OPEN_PORES 48  /* open-pore run starts kept per read in the record; n_open_pores is the true count */

typedef enum adb_status {
    ADB_OK = 0,
    ADB_ERR_CUDA = -1,          /* no device / CUDA runtime error                                             */
    ADB_ERR_ARG = -2,           /* invalid argument                                                            */
    ADB_ERR_MAD_ZERO = -3,      /* global MAD == 0: the reference raises ValueError (normalize.py:56-59)        */
    ADB_ERR_EMPTY_TRACE = -4,   /* a read has no downscaled sample: the reference raises ValueError (llr.py:136)
                                   outside any try and loses the minibatch (combined.py:145-211)              */
    ADB_ERR_UNSUPPORTED = -5,   /* configuration outside the built scope (e.g. windows larger than the build caps)  */
    ADB_ERR_OVERFLOW = -6       /* a record's open-pore list is longer than ADB_MAX_OPEN_PORES and its overflow row
                                   (adb_open_pores_host) was not supplied: nothing is ever truncated silently     */
} adb_status;

/* signal element types */
#define ADB_SIG_F32 0 /* calibrated pA, float32, dense [n_reads, m] row-major, NaN-padded (file_proc.py:160-175) */
#define ADB_SIG_I16 1 /* raw ADC int16, ragged: read i occupies [offsets[i], offsets[i+1]) of the blob         */

/* primary method codes (config/sig_proc.py:192-208) */
#define ADB_METHOD_LLR 0
#define ADB_METHOD_CNN 1
#define ADB_METHOD_START_PEAK 2

/* Flattened SigProcConfig (adapted/config/sig_proc.py:22-221).  Open range ends are +-inf. */
typedef struct adb_config {
    /* [core] */
    int32_t max_obs_trace, min_obs_adapter, max_obs_adapter, min_obs_polya, downscale_factor;
    int32_t primary_method;
    double sig_norm_outlier_thresh;
    /* [llr_boundaries] */
    double adapter_peak_prominence, adapter_peak_rel_height;
    int32_t adapter_peak_width;
    /* [cnn_boundaries] */
    int32_t polya_cand_k, fallback_to_llr_short_reads;
    /* [mvs_polya] */
    int32_t mvs_detect_check, mvs_detect_overwrite, search_window, pA_mean_window, pA_var_window;
    int32_t median_shift_window, polyA_window, pA_mean_range_empty, pA_mean_scale_range_empty;
    double pA_mean_range[2], pA_var_range[2], median_shift_range[2], polyA_med_range[2], polyA_local_range[2];
    double pA_mean_scale_range[2];
    /* [real_range] */
    int32_t detect_open_pores, real_signal_check, mean_window, max_obs_local_range;
    double mean_start_range[2], mean_end_range[2], local_range[2], adapter_mad_range[2];
    /* [med_shift] */
    int32_t detect_med_shift, med_shift_window;
    double med_shift_range[2];
    /* [rna_start_peak] */
    int32_t sp_downscale_factor, start_peak_max_idx, sp_offset1, sp_offset2;
    double open_pore_pa;
    int32_t sig_preload_size, _pad;
} adb_config;

/* fail_code values: the exact strings of combined.py:396-580 are produced by the host mirror */
enum adb_fail_code {
    ADB_FAIL_NONE = 0,
    ADB_FAIL_NO_ADAPTER = 1,        /* "No adapter detected (primary)"                     combined.py:396 */
    ADB_FAIL_ADAPTER_MAD = 2,       /* "adapter MAD check failed"                          combined.py:409 */
    ADB_FAIL_OPEN_PORE = 3,         /* "Open pore too close to boundary"                   combined.py:423 */
    ADB_FAIL_REAL_RANGE = 4,        /* "Real signal check failed"                          combined.py:439 */
    ADB_FAIL_NO_POLYA = 5,          /* "No polya detected (primary)"                       combined.py:444 */
    ADB_FAIL_MVS_NOT_ENOUGH = 6,    /* "MVS polya check failed: not enough signal"         combined.py:495 */
    ADB_FAIL_MVS_CHECKS = 7,        /* "MVS polya check failed: <names from mvs_fail_mask>" combined.py:515 */
    ADB_FAIL_MVS_NO_ADAPTER = 8,    /* "No adapter detected in range (mvs_detect)"         combined.py:542 */
    ADB_FAIL_MED_SHIFT = 9,         /* "Median shift check failed"                         combined.py:580 */
    ADB_FAIL_EXC_PA_MEAN_RANGE = 20,/* ValueError("pA_mean_range is not specified")        combined.py:462 */
    ADB_FAIL_EXC_TOPK_NONE = 21,    /* TypeError: 'NoneType' object is not iterable         combined.py:464 */
    ADB_FAIL_EXC_EMPTY_TRACE = 22,  /* ValueError from the hail-mary trace on an empty slice combined.py:277 */
    ADB_FAIL_EXC_SLICE_INDEX = 23,  /* TypeError: slice indices must be integers ... (start-peak, pandas)    */
    ADB_FAIL_EXC_MAD_ZERO = 24      /* ValueError("MAD normalization failed: scale is 0") in the hail mary   */
};

/* valid bits: which optional groups of the record are set (unset == None in DetectResults) */
#define ADB_V_ADAPTER_STATS (1u << 0)
#define ADB_V_POLYA_STATS (1u << 1)
#define ADB_V_RNA_STATS (1u << 2)
#define ADB_V_MVS (1u << 3)
#define ADB_V_REAL_MEANS (1u << 4)
#define ADB_V_REAL_RANGE (1u << 5)
#define ADB_V_OPEN_PORES (1u << 6)
#define ADB_V_MED_SHIFT (1u << 7)
#define ADB_V_CAND (1u << 8)
#define ADB_V_START_PEAK (1u << 9)
#define ADB_V_SP_OPEN_PORE (1u << 10)
#define ADB_V_FIELDS (1u << 11) /* cleared for reads that died on an exception: every field but fail is None */
/* mvs_detect_overwrite branch (combined.py:517-562, mean_var_shift_polyA_detect_at_loc mvs.py:181-338) */
#define ADB_V_MVS_ADAPTER_END (1u << 12) /* mvs_adapter_end is set                                              */
#define ADB_V_TO_EARLY_STOP (1u << 13)   /* mvs_llr_polya_end_to_early_stop = True                              */
#define ADB_V_POLYA_NONE (1u << 14)      /* polya_end became trace_early_stop_pos, which v0.2.4 never sets: None */

/* Fixed-layout result record, one per read (container_types.py:22-94 DetectResults). 512 bytes. */
typedef struct adb_record {
    int32_t success, fail_code, mvs_fail_mask;
    uint32_t valid;
    int32_t signal_len, preloaded;
    int32_t adapter_start, adapter_end, polya_end;    /* validated coordinates (combined.py:603-604,626) */
    int32_t primary_adapter_end, primary_polya_end;   /* {llr,cnn,start_peak}_{adapter,polya}_end (590-593) */
    int32_t mvs_adapter_end;
    int32_t n_cand, cand[ADB_MAX_CAND];               /* polya_candidates */
    int32_t n_open_pores, open_pores[ADB_MAX_OPEN_PORES];
    int32_t sp_idx, sp_next_idx, sp_open_pore_idx, sp_flag; /* start_peak_* (333-338); sp_flag 1/2 = type */
    float sp_pa, sp_next_pa;
    double stats[3][4];  /* adapter / polya / rna_preloaded x mean, std, med, mad (signal_partitions.py:81-96) */
    double mvs[5];       /* mvs_detect_{mean_at_loc,var_at_loc,polya_med,polya_local_range,med_shift}          */
    double real[3];      /* real_adapter_{mean_start,mean_end,local_range}                                      */
    double med_shift;    /* adapter_rna_median_shift                                                            */
    uint8_t _reserved[8];
} adb_record;

/* ---- library ---------------------------------------------------------------------------------------- */
int adb_abi_version(void);
const char *adb_last_error(void);
int adb_device_count(void);
int adb_record_size(void);
int adb_config_size(void);

/* Opaque per-device context: owns the scratch arena, pinned staging buffers and two CUDA streams. */
typedef struct adb_ctx adb_ctx;
int adb_ctx_create(int device, adb_ctx **out);
void adb_ctx_destroy(adb_ctx *ctx);
/* number of kernels this context has launched so far (bench.py: gpu_launches) */
int64_t adb_ctx_launch_count(const adb_ctx *ctx);
/* Tuning switches that never change results.  "exact_global_select" = 1: always take the multi-pass radix select
 * for the minibatch-global median / MAD (normalize.py:15-22) instead of the sampled one-pass select.
 * "no_fast_validate" = 1: int16 reads go through the histogram-based validate kernel only (A/B testing).
 * "host_zstd" = 1: adb_detect_files decompresses the zstd frames of VBZ containers on the host (libzstd) instead of
 * on the GPU (A/B testing; the reference of the device path). */
int adb_ctx_set_option(adb_ctx *ctx, const char *name, int value);
/* Diagnostics of the most recent call (synchronises the device).  "global_select_fallbacks": minibatches the sampled
 * select handed to the exact multi-pass select; "validate_handovers": reads the counting-based validate kernel left
 * to the histogram-based one (both for the last pass of at most 256 minibatches); "zstd_host_frames": zstd frames
 * the last adb_detect_files call decompressed on the host.  -1: unknown name / error. */
int64_t adb_ctx_query(adb_ctx *ctx, const char *name);

/* ---- minibatch detection ---------------------------------------------------------------------------- */
/*
 * One description of a batch of reads.  `n_batches` consecutive groups of `batch_size` reads (the last may be
 * short) are independent minibatches: the LLR path normalises with ONE median/MAD per minibatch
 * (combined.py:128-132) and the CNN path couples reads of a minibatch through a flattened peak search
 * (cnn.py:140), so the reference's minibatch (default 1000 reads, parser.py:95-99) is the unit of work.
 */
typedef struct adb_batch {
    const void *signal;          /* f32 dense matrix or i16 blob (host or device, see the function)   */
    int32_t sig_type;            /* ADB_SIG_F32 | ADB_SIG_I16                                         */
    int32_t n_reads;
    int32_t m;                   /* preload window: row length (F32) / max samples per read (I16)     */
    int32_t batch_size;          /* reads per minibatch                                               */
    const int64_t *offsets;      /* I16: [n_reads+1] element offsets into the blob; F32: NULL         */
    const int32_t *full_lens;    /* [n_reads] untruncated read lengths (file_proc.py:161,171)        */
    const float *calib_offset;   /* I16: [n_reads] pA = (adc + offset) * scale in float32; F32: NULL  */
    const float *calib_scale;
} adb_batch;

/*
 * Drop-in for combined_detect_llr2(batch_of_signals, full_signal_lens, spc)   adapted/detect/combined.py:122-227
 *          and combined_detect_cnn(batch, lens, model, spc)                   adapted/detect/combined.py:230-309
 *          and combined_detect_start_peak(batch, lens, spc)                   adapted/detect/combined.py:312-355
 * selected by cfg->primary_method.  `cnn_weights` (CNN only) is the model's state dict flattened in the order
 * 0.weight[64,1,7] 0.bias[64] 2.weight[64,64,7] 2.bias[64] 4.weight[64,64,7] 4.bias[64] 6.weight[64,2,7] 6.bias[2]
 * (58 882 floats, adapted/detect/cnn.py:16-52).  `batch_status` (optional, [n_batches]) receives the per-minibatch
 * adb_status (where the reference raises outside its per-read try and loses the minibatch).
 * Supported preload windows (batch->m = sig_preload_size): any m up to 131 072 samples, for ADB_SIG_I16 and
 * ADB_SIG_F32 alike, here and in adb_detect_dev, adb_detect_pipelined_host, adb_detect_pipelined_svb_host and
 * adb_detect_files.  Windows too long for a kernel's shared-memory layout take a variant that reads the signal from
 * global memory (same records).  Ceilings that remain return ADB_ERR_UNSUPPORTED with adb_last_error() naming them:
 * the 16-bit working-set indices of the CNN top-k (about 437 000 samples at downscale factor 10), the CNN path's
 * hail-mary LLR trace and the LLR primary trace in shared memory (both above about 21 000 downscaled points, i.e.
 * m / downscale_factor; far above 131 072 samples at the shipped downscale factors).
 */
int adb_detect_host(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                    adb_record *out_records, int32_t *batch_status);
/* Same, all pointers inside `batch`, `cnn_weights`, `out_records`, `batch_status` are DEVICE pointers. */
int adb_detect_dev(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                   adb_record *out_records, int32_t *batch_status, void *cuda_stream);

/*
 * Streaming ingest (replaces the producer thread + process pool of adapted/file_proc.py:143-214,738-784 for one
 * GPU): HOST (ideally pinned) ragged int16 reads are cut into chunks of `chunk_batches` minibatches; the H2D
 * copy of chunk i+1 overlaps the kernels of chunk i, records are copied back per chunk.  Synchronous on return.
 */
int adb_detect_pipelined_host(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                              adb_record *out_records, int32_t *batch_status, int32_t chunk_batches);

/* Per-kernel-class device timing (CUDA events around every launch; used by bench.py for the roofline):
 * class 0 streaming pass of the minibatch-global median / MAD (multi-pass histogram kernels when forced),
 * 1 its sample / plan / finish kernels (scan kernels of the multi-pass select when forced), 2 validate kernel
 * (counting-based for int16 reads, histogram-based otherwise), 3 LLR-primary kernel, 4 moving-statistics kernels,
 * 5 the CNN's convolution kernels (tcgen05 layers 2 / 3; FP32-pipe kernels + convT when selected), 6 start-peak kernels
 * and the CNN's pre- / post-processing (prep, peak search, top-k), 7 hand-over kernels (what the fast paths pass on
 * to the general kernels, incl. the FP32-pipe redo of reads outside the tensor-core kernels' fp16 range).
 * adb_ctx_get_timing fills out[16] = {ms, launches} x 8; call it after synchronising the stream. */
int adb_ctx_set_timing(adb_ctx *ctx, int on);
int adb_ctx_get_timing(adb_ctx *ctx, double *out);

/* ---- kernel-level entry points (differential tests against the Cython module) -------------------------- */
/*
 * Drop-in for c_llr_trace(raw_signal, start, end, min_obs, border_trim, stride, adapter_early_stopping,
 *   adapter_early_stop_window, adapter_early_stop_stride, polya_early_stopping, polya_early_stop_window,
 *   polya_early_stop_stride, return_c_c2)                                  adapted/detect/_c_llr.pyx:202-236
 * for `n_traces` signals at once (signal i = signals[sig_offsets[i] .. sig_offsets[i+1]), float64, HOST).
 * params[i*11 .. i*11+11) = start,end,min_obs,border_trim,stride,aes,aes_window,aes_stride,pes,pes_window,pes_stride.
 * gains / c / c2 (c, c2 optional) use the same offsets.
 */
int adb_llr_trace_host(adb_ctx *ctx, const double *signals, const int64_t *sig_offsets, int32_t n_traces,
                       const int64_t *params, double *gains, double *c, double *c2);

/*
 * Drop-in for the legacy three-split detectors (no caller inside the reference; library-level operators)
 *   c_llr_detect_adapter(raw_signal, min_obs_adapter, border_trim)                      adapted/detect/_c_llr.pyx:239-288
 *   c_llr_detect_adapter_polya(raw_signal, min_obs_adapter, border_trim, min_obs_polya) adapted/detect/_c_llr.pyx:290-363
 * (both on _best_split, _c_llr.pyx:40-64) for `n_signals` float64 signals at once (HOST buffers, offsets as above).
 * params[i*3 .. i*3+3) = min_obs_adapter, border_trim, min_obs_polya (< 0: adapter only, polya_end stays 0).
 * out[i*4 .. i*4+4) = adapter_start, adapter_end, polya_end, length of the tuple the reference returns (2: the
 * "empty signal" early return of either function, else 3).
 */
int adb_llr_detect_host(adb_ctx *ctx, const double *signals, const int64_t *sig_offsets, int32_t n_signals,
                        const int64_t *params, int64_t *out);

/*
 * Peak picking on given traces (kernel-level test entry for the scipy.signal.find_peaks subset and the corrections
 * built on it; HOST buffers, trace i = traces[offsets[i] .. offsets[i+1]), float64, at most 4096 points each).
 * params[i*8 .. i*8+8) (float64) = mode, distance, prominence, width, rel_height, want, nan_to_num, unused:
 *   mode 0  find_peaks(trace, distance, prominence, width, rel_height): the first `want` (<= 32) peaks in ascending
 *           order (scipy/signal/_peak_finding.py:729-1010 as used at llr.py:189,218,444; nan_to_num as llr.py:445)
 *   mode 1  adapter_end_from_trace (llr.py:204-259): LLRTrace support, find_peaks(width, prominence * nanstd,
 *           rel_height), correct_for_plateau, correct_for_split_peak -> cands[0] or -1 (no candidate)
 *   mode 2  detect_full_polya_trace_peak_with_spike (llr.py:406-479) -> index or 0
 * out[i*33] = number of values, out[i*33 + 1 ..] the values.
 */
int adb_find_peaks_host(adb_ctx *ctx, const double *traces, const int64_t *offsets, int32_t n_traces, const double *params,
                        int32_t *out);

/* Minibatch-global median / MAD of normalize_signal (adapted/detect/normalize.py:15-22,54), HOST buffers. */
int adb_global_med_mad_host(adb_ctx *ctx, const adb_batch *batch, int32_t max_obs_trace, float *med_mad /*[n_batches*2]*/);

/* mean-pool downscale of efficient_average_pooling (adapted/detect/downscale.py:4-41) on raw pA, HOST buffers:
 * out[n_reads, ceil(m / factor)] float32 (NaN where the block has a NaN). */
int adb_downscale_host(adb_ctx *ctx, const adb_batch *batch, int32_t col0, int32_t factor, float *out);

/* CNN scores of BoundariesCNN (adapted/detect/cnn.py:16-52,85-98) on prepared inputs x[n, L] -> scores[n, 2, L_out] */
int adb_cnn_scores_host(adb_ctx *ctx, const float *x, int32_t n, int32_t L, const float *cnn_weights, float *scores);

/* ---- streaming poly(A) detector (SURVEY.md row f4) --------------------------------------------------------- */
/* StreamingConfig (adapted/config/sig_proc.py:140-158); open range ends are +-inf */
typedef struct adb_stream_config {
    int32_t min_obs_adapter, min_obs_post_loc, search_increment_step;
    int32_t pA_mean_window, pA_var_window, median_shift_window, polyA_window, _pad;
    double pA_mean_range[2], pA_var_range[2], median_shift_range[2], polyA_med_range[2], polyA_local_range[2];
} adb_stream_config;
/*
 * Drop-in for mean_var_shift_polyA_detect(calibrated_signal, params)            adapted/detect/mvs.py:341-426
 * (read-until / streaming poly(A) detection on an accumulating signal cache; no caller inside the reference) for
 * every read of `batch` at once (HOST buffers; read i is its first min(full_lens[i], m) samples, I16 or F32 form).
 * polya_start[i] = the detected poly(A) start or 0.
 */
int adb_mvs_stream_detect_host(adb_ctx *ctx, const adb_batch *batch, const adb_stream_config *cfg, int32_t *polya_start);

/*
 * Read-until sessions of the same detector: the caller keeps asking "where does the poly(A) start in what this
 * channel has delivered so far?" while the cache grows chunk by chunk.  A session holds `n_slots` slots (one per
 * channel), each the int16 ADC cache (at most `max_samples` samples) of the read on it plus that read's calibration,
 * on the context's device; pushes run on the context's stream.  The cache is never staged in shared memory, so
 * max_samples is not bounded by the stateless call's window.
 *
 * After a push, every pushed slot k returns
 *   polya_start[k]  exactly what mean_var_shift_polyA_detect(calibrate(cache), cfg) returns on the slot's whole cache
 *                   (adb_mvs_stream_detect_host on the same samples), pA = (float32(adc) + offset) * scale;
 *   settled[k]      1 when no later sample can change that answer: an acceptance whose windows are complete, or a full
 *                   cache (samples beyond max_samples are dropped).  Chunks for a settled read are ignored.
 * Per push, only the appended samples enter the moving statistics, and the search loop resumes after its last final
 * decision (adb_stream_session.cuh).
 */
typedef struct adb_stream_session adb_stream_session;
/* ADB_ERR_ARG for n_slots < 1 or max_samples < 1, ADB_ERR_UNSUPPORTED for the configurations that
 * adb_mvs_stream_detect_host refuses.  The context must outlive the session. */
int adb_stream_session_create(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots, int32_t max_samples,
                              adb_stream_session **out);
void adb_stream_session_destroy(adb_stream_session *s);
/* entry k: reset[k] != 0 starts a new read on slots[k] (cache emptied, calibration taken from calib_offset[k] /
 * calib_scale[k]), then adc[chunk_offsets[k] .. chunk_offsets[k+1]) is appended.  HOST buffers, synchronous.
 * reset == NULL: no entry resets (calib_* may then be NULL).  Zero-length chunks are legal and return the current
 * answer.  ADB_ERR_ARG, with the session unchanged, for a slot out of range or twice in one push, decreasing offsets,
 * an append to a slot that was never reset, or a reset with a non-finite offset or a non-finite or non-positive
 * scale. */
int adb_stream_session_push(adb_stream_session *s, int32_t n, const int32_t *slots, const int64_t *chunk_offsets,
                            const int16_t *adc, const uint8_t *reset, const float *calib_offset,
                            const float *calib_scale, int32_t *polya_start, uint8_t *settled);
/*
 * Float32 sessions: the same detector on caches of calibrated float32 pA, the input of mean_var_shift_polyA_detect
 * itself (read-until clients that receive calibrated chunks).  polya_start[k] is exactly what
 * adb_mvs_stream_detect_host returns on the slot's whole cache as ADB_SIG_F32; `settled` and the handling of settled
 * reads and of max_samples are those of the int16 session.  adb_stream_session_destroy frees either kind.
 */
/* as adb_stream_session_create; the cache takes n_slots * max_samples * 4 bytes of device memory */
int adb_stream_session_create_f32(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots, int32_t max_samples,
                                  adb_stream_session **out);
/* entry k: reset[k] != 0 starts a new read on slots[k] (cache emptied; no calibration), then
 * pa[chunk_offsets[k] .. chunk_offsets[k+1]) is appended.  HOST buffers, synchronous.  ADB_ERR_ARG, with the session
 * unchanged, for the errors of adb_stream_session_push, for a non-finite sample (NaN, +-inf) anywhere in the pushed
 * chunks (also in chunks that are ignored or clipped), and for a float32 push on an int16 session;
 * adb_stream_session_push refuses an int16 push on a float32 session the same way. */
int adb_stream_session_push_f32(adb_stream_session *s, int32_t n, const int32_t *slots, const int64_t *chunk_offsets,
                                const float *pa, const uint8_t *reset, int32_t *polya_start, uint8_t *settled);
/*
 * Device-push sessions: the same sessions for clients that hold their chunks on the GPU.  A push reads its entries and
 * chunks from device memory and writes its answers to device memory; all its work is enqueued on the caller's stream,
 * with no host synchronise and no allocation, so pushes overlap the caller's own kernels and can be captured in a
 * CUDA graph.  Answers and refusals are exactly those of the host push.  Host pushes (adb_stream_session_push /
 * _push_f32) refuse a device-push session, and adb_stream_session_push_dev refuses the other sessions.
 */
/* as adb_stream_session_create / _create_f32 with sig_type ADB_SIG_I16 / ADB_SIG_F32 (anything else: ADB_ERR_ARG).
 * Allocates everything a push needs (cache, mask, slot state, and entry and validation scratch for n_slots entries);
 * adb_stream_session_destroy frees it. */
int adb_stream_session_create_dev(adb_ctx *ctx, const adb_stream_config *cfg, int32_t n_slots, int32_t max_samples,
                                  int32_t sig_type, adb_stream_session **out);
/*
 * One push, every pointer a DEVICE pointer, asynchronous on `cuda_stream` (a cudaStream_t; NULL is CUDA's default
 * stream).  The arguments mean what they mean for adb_stream_session_push / _push_f32: `samples` holds int16 ADC or
 * float32 pA as the session does, at least chunk_offsets[n] of them; calib_offset / calib_scale are NULL for float32.
 * polya_start (int32 [n]) and settled (uint8 [n]) receive what the host push returns, including the final answer of a
 * settled slot.  status (int32 [2]) receives {adb_status, reason}: {ADB_OK, 0} for an accepted push, {ADB_ERR_ARG,
 * reason} for a refused one, which changes neither the session nor polya_start / settled.
 * adb_stream_session_reason(reason) is the text adb_last_error() gives for the same refusal of the host push.
 * Everything that depends on the data is checked on the device, in stream order, before any state changes; the call
 * itself returns ADB_ERR_ARG, enqueueing nothing, only for a null handle, status or array pointer, a session that is
 * not a device-push session, n > n_slots (a valid push names each slot at most once), or a calibration given to a
 * float32 session.  Pushes to one session must be ordered on the device (one stream, or events between streams).
 */
int adb_stream_session_push_dev(adb_stream_session *s, int32_t n, const int32_t *slots, const int64_t *chunk_offsets,
                                const void *samples, const uint8_t *reset, const float *calib_offset,
                                const float *calib_scale, int32_t *polya_start, uint8_t *settled, int32_t *status,
                                void *cuda_stream);
/* the text of a refusal reason of adb_stream_session_push_dev's status[1]; NULL for 0 and unknown codes */
const char *adb_stream_session_reason(int32_t reason);

/* ---- result tables (SURVEY.md row f2) ---------------------------------------------------------------------- */
/*
 * Drop-in for save_detected_boundaries(processing_results, filename, save_fail_reasons)   adapted/output.py:26-51
 * (with ReadResult.to_summary_dict, adapted/container_types.py:112-120): the CSV text pandas writes for the reads
 * `sel[0..n_sel)` of `recs` (sel == NULL: the first n_sel records), byte for byte -- column order, per-column type
 * inference (an int column holding a None prints as float), round(3), numpy's str() of the candidate / open-pore
 * arrays, empty cells for None, `fail_reason` last and only if save_fail_reasons.  Pure host code, no device needed.
 * read_ids[i] belongs to recs[i].  Returns the number of bytes of the table; when that exceeds `cap` nothing useful
 * is in `out` and the call is to be repeated with a larger buffer (cap = 0, out = NULL sizes the table).
 */
int64_t adb_format_csv(const adb_record *recs, const int32_t *sel, int32_t n_sel, const char *const *read_ids,
                       int32_t primary_method, const char *llr_detect_log, int32_t save_fail_reasons, char *out,
                       int64_t cap);

/* Same with the overflow rows of the open-pore lists: records with n_open_pores > ADB_MAX_OPEN_PORES print the full
 * list op_pos[op_offsets[k] .. op_offsets[k + 1]) with k = op_index[i] (op_index: one entry per record of `recs`, -1 =
 * no row).  A record beyond the cap without a row of exactly n_open_pores entries makes both functions return
 * ADB_ERR_OVERFLOW (the reference prints the whole array, combined.py:412-419; nothing is truncated silently). */
int64_t adb_format_csv_ex(const adb_record *recs, const int32_t *sel, int32_t n_sel, const char *const *read_ids,
                          int32_t primary_method, const char *llr_detect_log, int32_t save_fail_reasons,
                          const int32_t *op_index, const int64_t *op_offsets, const int32_t *op_pos, char *out,
                          int64_t cap);

/*
 * find_open_pores(signal[adapter_start:adapter_end])                 adapted/detect/anomalies.py:15-35
 * in full for the reads sel[0..n_sel) of `batch` (HOST buffers) over the sample range [seg_begin[k], seg_end[k]) --
 * the overflow path of the fixed-size record: validate_boundaries scans [0, primary adapter_end)
 * (combined.py:411-419), the record keeps the first ADB_MAX_OPEN_PORES positions and the true count.
 * out_offsets[n_sel + 1] always receives the prefix sums of the list lengths; the positions (window coordinates) are
 * written only if cap >= out_offsets[n_sel] (call with cap = 0 to size the buffer).
 */
int adb_open_pores_host(adb_ctx *ctx, const adb_batch *batch, const int32_t *sel, int32_t n_sel,
                        const int32_t *seg_begin, const int32_t *seg_end, int64_t *out_offsets, int32_t *out_pos,
                        int64_t cap);

/* ---- compressed ingest (SURVEY.md row f1) -------------------------------------------------------------------- */
/*
 * VBZ-style compressed reads: what pod5 stores per signal chunk minus its zstd stage, i.e. svb16(zigzag(delta)) of
 * the int16 samples (pod5 c++/pod5_format/svb16; replaces the decode inside pod5's ReadRecord.signal that
 * yield_signals_from_pod5 calls, adapted/file_proc.py:165-175).  Read i's stream starts at comp[comp_offsets[i]]
 * (16-byte aligned): ceil(n / 8) key bytes (bit j % 8 of byte j / 8: 0 = one data byte, 1 = two, little endian), zero
 * padded to a multiple of 4, then the data bytes of the n = n_samples[i] <= m values; 16 bytes of slack follow the
 * last stream.  About 1.15 bytes per sample on nanopore signal instead of 2.
 */
typedef struct adb_svb_batch {
    const uint8_t *comp;
    const int64_t *comp_offsets; /* [n_reads + 1] */
    const int32_t *n_samples;    /* [n_reads] stored samples per read = min(full length, preload window)  */
    int32_t n_reads, m, batch_size, _pad;
    const int32_t *full_lens;
    const float *calib_offset, *calib_scale;
} adb_svb_batch;

/* svb16 + zig-zag + delta decode on the GPU, HOST buffers in and out (kernel-level test entry): out_adc receives the
 * reads back to back (read i at the exclusive prefix sum of n_samples). */
int adb_svb16_decode_host(adb_ctx *ctx, const adb_svb_batch *batch, int16_t *out_adc);
/*
 * adb_detect_pipelined_host for compressed reads: every chunk travels host -> device COMPRESSED (pinned host buffers
 * for asynchronous copies), is decoded by svb16_decode_kernel into the ragged int16 layout and detected; records
 * return per chunk.  Replaces producer thread + pod5 decode + process pool (file_proc.py:143-214,738-784) for one GPU.
 * ctx option "pipeline_copy_only" = 1 skips the kernels (bench.py: the box's host -> device ceiling for these chunks).
 */
int adb_detect_pipelined_svb_host(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                                  adb_record *out_records, int32_t *batch_status, int32_t chunk_batches);

/* ---- VBZ ingest: the zstd stage on the GPU (adb_zstd.cuh) ------------------------------------------------------ */
/*
 * zstd decode on the GPU (RFC 8878 frames without dictionaries), HOST buffers (kernel-level test entry): frame i =
 * src[src_offsets[i] .. src_offsets[i + 1]) decodes into the slot dst[dst_offsets[i] .. dst_offsets[i + 1]).
 * status[i] = the decoded size, or a negative ADB_ZSTD_E_* code; a refused frame leaves everything outside its slot
 * untouched.  Bytes of a slot past the decoded size are unspecified (the decoder parks literals there).  Every frame
 * is decoded on the device, including the ones adb_detect_files would leave to the host.
 */
#define ADB_ZSTD_E_TRUNCATED (-1) /* frame ends before its last block, or a section runs past its block      */
#define ADB_ZSTD_E_MAGIC (-2)     /* not a zstd frame (skippable frames included)                             */
#define ADB_ZSTD_E_RESERVED (-3)  /* reserved bit, block type or sequence mode bits set                       */
#define ADB_ZSTD_E_DICT (-4)      /* dictionary ID other than 0                                               */
#define ADB_ZSTD_E_DST_SIZE (-5)  /* output past the slot, or a block past the block maximum                  */
#define ADB_ZSTD_E_OFFSET (-6)    /* match offset beyond the bytes produced or the window                     */
#define ADB_ZSTD_E_SIZE (-7)      /* decoded size differs from the frame's content size                       */
#define ADB_ZSTD_E_CHECKSUM (-8)  /* XXH64 content checksum mismatch                                          */
#define ADB_ZSTD_E_CORRUPT (-9)   /* a table description or bitstream RFC 8878 declares corrupt               */
#define ADB_ZSTD_E_TRAILING (-10) /* bytes left over behind the frame                                         */
int adb_zstd_decompress_host(adb_ctx *ctx, const uint8_t *src, const int64_t *src_offsets, int32_t n, uint8_t *dst,
                             const int64_t *dst_offsets, int32_t *status);
/*
 * adb_detect_pipelined_svb_host for VBZ reads (pod5's signal form): batch->comp holds one zstd frame per read
 * (comp_offsets delimit the frames; no alignment or slack needed).  Frames travel host -> device as they are and go
 * through zstd_decode_kernel, svb16_decode_kernel and detection.  Every frame must hold a content size of at most the
 * worst-case stream of m samples and no dictionary (ADB_ERR_UNSUPPORTED otherwise); a frame the device refuses fails
 * the call with ADB_ERR_ARG.  "pipeline_copy_only" skips the kernels.
 */
int adb_detect_pipelined_vbz_host(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                                  adb_record *out_records, int32_t *batch_status, int32_t chunk_batches);

/* ---- file level (SURVEY.md row f1): containers -> GPU -> boundary tables, all stages overlapped ------------- */
/*
 * Drop-in for the part of run_detect between the reader and the CSV files for ONE GPU
 *   producer thread yield_signals_from_pod5        adapted/file_proc.py:143-214
 *   process pool + worker seam                      adapted/file_proc.py:217-266, 738-784
 *   saver threads / save_detected_boundaries        adapted/file_proc.py:312-457, adapted/output.py:26-51
 * on "ADBSIG02" signal containers (adapted_b200/ingest.py:write_container_v2: per read the svb16 stream of its first
 * min(length, preload window) samples, optionally one zstd frame per read = pod5's VBZ; or raw int16).  A reader
 * thread fills a ring of pinned host slots (chunks of `chunk_batches` minibatches, cut in file order across file
 * boundaries), this thread copies / decodes / detects on alternating contexts, a writer thread splits the records
 * into the pass / fail lists in arrival order and formatter threads write <out_dir>/boundaries/
 * detected_boundaries_<i>.csv and <out_dir>/failed_reads/failed_reads_<i>.csv (batch_size_output reads per table,
 * numbering from bidx_pass / bidx_fail: `adapted continue`, file_proc.py:97-140).
 */
typedef struct adb_file_job {
    const char *const *paths;
    int32_t n_paths;
    int32_t minibatch_size;        /* reads per minibatch (parser.py:95-99: 1000)                                  */
    const uint8_t *const *keep;    /* optional [n_paths]: per file one byte per read, 0 = skip (selection / continue) */
    const char *out_dir;
    int32_t batch_size_output;     /* reads per table (parser.py:87-93: 4000)                                      */
    int32_t chunk_batches;         /* minibatches per pipeline chunk (0: 16)                                       */
    int32_t bidx_pass, bidx_fail;  /* first table indices                                                          */
    int32_t n_copy_threads, n_format_threads; /* 0: defaults                                                       */
    int32_t write_csv, _pad;       /* 0: detection only (records are dropped; statistics still filled)             */
} adb_file_job;
typedef struct adb_file_stats {
    int64_t reads, pass, fail, lost, files, comp_bytes, h2d_bytes;
    double seconds, read_s, gpu_wait_s, write_s; /* wall time of the call; busy time of the reader / writer stages */
} adb_file_stats;
int adb_detect_files(adb_ctx *ctx, const adb_file_job *job, const adb_config *cfg, const float *cnn_weights,
                     adb_file_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* ADAPTED_B200_H */
