// validate_boundaries (combined.py:358-631) downstream of the order statistics, written once for every validation kernel.
//
// validate_fast_kernel (adb_vfast.cuh, counting passes) and validate_hist_kernel (adb_vhist.cuh, tensor-core
// histograms) find the statistics of the same twelve sample ranges their own way and hand them over in a VcStats; the
// functions here decode the read's inputs, lay out the ranges, run the checks (SURVEY A.8) and write the record.
// validate_cand_kernel and validate_boundaries_cta (adb_validate.cuh) share the MVS helpers and the record writers.
//
// Pure per-thread code: no barriers, no shared memory of its own, each kernel keeps its own sync scope around the calls
// (validate_fast_kernel runs the checks on thread 0, validate_hist_kernel on warp 0).
#pragma once
#include "adb_common.cuh"
#include "adb_gsample.cuh"

struct VfastArgs {
    BatchDev B;
    const int *given;           // [n_reads][given_stride] = adapter_end, polya_end(= topk[0]), topk[1..]
    int given_stride;
    int given_ntopk;            // entries per read when ntopk_per_read == nullptr (-1: None)
    const int *ntopk_per_read;
    int mode;                   // ADB_METHOD_*
    int win_bytes;              // capacity of the staged window (bytes)
    adb_record *out;
    const int *batch_status;
    const float *pre_var, *pre_mean;  // compact pools of precomputed moving statistics (mvs_series_kernel)
    const long long *pre_off;
    const int *pre_meta;
    const float *series_med;    // [n_reads][2] medians of the two series of the row (series_median_kernel)
    unsigned char *done;        // [n_reads], zeroed before the launch; 1 = record written by this kernel,
                                // 2 = record written with the FIRST poly(A) candidate's outcome, further candidates pending
    int cand_followup;          // 1: validate_cand_kernel runs behind this kernel (CNN path with several candidates)
};

// ---- numpy mean / variance of a short segment ---------------------------------------------------------------------
// float32 np.mean and np.var (numpy _var: mean, x - mean, x * x, pairwise sum / n) of x(0) .. x(n - 1), one thread
template <class F>
__device__ __forceinline__ float np_mean_f32(F x, int n) { return __fdiv_rn(np_sum_f32(x, n), (float)n); }
template <class F>
__device__ __forceinline__ float np_var_f32(F x, int n, float mean) {
    return __fdiv_rn(np_sum_f32([&](int i) { const float d = __fsub_rn(x(i), mean); return __fmul_rn(d, d); }, n), (float)n);
}

// ---- MVS check helpers (mvs.py:45-158, combined.py:447-515) --------------------------------------------------------
// bounds of the poly(A) mean: the configured range, or the scale range times the adapter median when that is empty;
// false when both are empty (the reference raises)
__device__ __forceinline__ bool vc_pa_mean_bounds(const adb_config &cfg, float a_med, double mr[2]) {
    mr[0] = cfg.pA_mean_range[0];
    mr[1] = cfg.pA_mean_range[1];
    if (!cfg.pA_mean_range_empty) return true;
    if (cfg.pA_mean_scale_range_empty) return false;
    mr[0] = __dmul_rn(cfg.pA_mean_scale_range[0], (double)a_med);
    mr[1] = __dmul_rn(cfg.pA_mean_scale_range[1], (double)a_med);
    return true;
}

// bit i: check i failed (mean, var, median, local range, median shift)
__device__ __forceinline__ int vc_mvs_mask(const adb_config &cfg, const double v[5], const double mr[2]) {
    int mask = 0;
    if (!in_range_d(v[0], mr)) mask |= 1;
    if (!in_range_d(v[1], cfg.pA_var_range)) mask |= 2;
    if (!in_range_d(v[2], cfg.polyA_med_range)) mask |= 4;
    if (!in_range_d(v[3], cfg.polyA_local_range)) mask |= 8;
    if (!in_range_d(v[4], cfg.median_shift_range)) mask |= 16;
    return mask;
}

// fail reason of a failed candidate: combined.py:492-495 keys on the mean value (0: the check returned early)
__device__ __forceinline__ void vc_mvs_fail(double mean, int mask, int &fail, int &fail_mask) {
    if (mean == 0.0) { fail = ADB_FAIL_MVS_NOT_ENOUGH; fail_mask = 0; }
    else { fail = ADB_FAIL_MVS_CHECKS; fail_mask = mask; }
}

// ---- the outcome and the record ------------------------------------------------------------------------------------
struct VcOut {
    bool success;
    bool exception;  // the reference raises inside validate_boundaries: exception record
    bool defer;      // validate_kernel redoes the read from scratch
    bool followup;   // validate_cand_kernel finishes the read (further poly(A) candidates)
    int fail, fail_mask;
    uint32_t valid;
    int a_start, n_open;
    double mvs[5], real[3], med_shift;
};

__device__ __forceinline__ VcOut vc_out(int a_start) {  // before the first check
    VcOut o;
    o.success = true; o.exception = false; o.defer = false; o.followup = false;
    o.fail = ADB_FAIL_NONE; o.fail_mask = 0;
    o.valid = ADB_V_FIELDS;
    o.a_start = a_start; o.n_open = 0;
    for (int i = 0; i < 5; i++) o.mvs[i] = 0.0;
    for (int i = 0; i < 3; i++) o.real[i] = 0.0;
    o.med_shift = 0.0;
    return o;
}

// combined.py:225-226 / 304-305 / 350-351: DetectResults(success=False, fail_reason=str(e)), all else None.  One thread.
__device__ __forceinline__ void vc_write_exception(adb_record *rec, int fail, int full_len, int size) {
    rec->success = 0; rec->fail_code = fail; rec->mvs_fail_mask = 0; rec->valid = 0;
    rec->signal_len = full_len; rec->preloaded = min(full_len, size);
}

// the record of a validated read; `cand` holds the n_topk poly(A) candidates.  One thread.
__device__ __forceinline__ void vc_write_record(adb_record *rec, const VcOut &o, const double st[3][4], int full_len, int size,
                                                int a_end, int polya_end, int primary_a_end, int primary_polya_end,
                                                int mvs_a_end, int n_topk, const int *cand) {
    rec->success = o.success ? 1 : 0;
    rec->fail_code = o.fail;
    rec->mvs_fail_mask = o.fail_mask;
    rec->valid = o.valid | (n_topk >= 0 ? ADB_V_CAND : 0);
    rec->signal_len = full_len;
    rec->preloaded = min(full_len, size);
    rec->adapter_start = o.a_start;
    rec->adapter_end = a_end;
    rec->polya_end = polya_end;
    rec->primary_adapter_end = primary_a_end;
    rec->primary_polya_end = primary_polya_end;
    rec->mvs_adapter_end = mvs_a_end;
    rec->n_cand = max(n_topk, 0);
    for (int t = 0; t < ADB_MAX_CAND; t++) rec->cand[t] = (t < n_topk) ? cand[t] : 0;
    rec->n_open_pores = o.n_open;
    for (int p = 0; p < 3; p++) for (int q = 0; q < 4; q++) rec->stats[p][q] = st[p][q];
    for (int i = 0; i < 5; i++) rec->mvs[i] = o.mvs[i];
    for (int i = 0; i < 3; i++) rec->real[i] = o.real[i];
    rec->med_shift = o.med_shift;
}

__device__ __forceinline__ void vc_zero_record(adb_record *rec) {  // CTA-strided
    for (int w = threadIdx.x; w < (int)(sizeof(adb_record) / 4); w += blockDim.x) ((uint32_t *)rec)[w] = 0;
}

// ---- the speculative kernels (validate_fast_kernel, validate_hist_kernel) -------------------------------------------
// The start of every read: a read of a lost minibatch gets a zero record (the host raises), a read without int16
// samples and a usable calibration is left to validate_kernel.  False for both.
__device__ __forceinline__ bool vc_read_start(const VfastArgs &A, int r, ReadSrc &src) {
    if (A.batch_status[r / A.B.batch_size] != ADB_OK) {
        vc_zero_record(A.out + r);
        if (threadIdx.x == 0) A.done[r] = 1;
        return false;
    }
    src = make_src(A.B, r);
    return src.i16 != nullptr && src.cscale > 0.0f && isfinite(src.cscale) && isfinite(src.coff);
}

struct VcIn {  // per-read inputs of the checks
    const int *g;              // the read's row of `given`
    int full_len, size;
    float coff, cscale;
    int a_end, pe_best, n_topk, pe0, topk1;
    bool mvs_geom;             // the MVS check of the first candidate gets past its early return
    bool win_var, win_mean;    // its variance / mean are medians of moving statistics (else: of the short segment)
    float smed_var, smed_mean; // those medians (series_median_kernel)
};

// false: the moving statistics of the read are not precomputed, validate_kernel takes the read
__device__ __forceinline__ bool vc_inputs(const VfastArgs &A, const adb_config &cfg, int r, const ReadSrc &src, VcIn &I) {
    const int *g = A.given + (size_t)r * A.given_stride;
    I.g = g;
    I.full_len = A.B.full_lens[r];
    I.size = src.n;
    I.coff = src.coff; I.cscale = src.cscale;
    I.a_end = g[0]; I.pe_best = g[1];
    I.n_topk = A.ntopk_per_read ? A.ntopk_per_read[r] : A.given_ntopk;
    I.pe0 = (I.n_topk >= 1) ? g[1] : 0;
    I.topk1 = (I.n_topk >= 2) ? g[2] : 0;
    const int a_end = I.a_end, pe0 = I.pe0;
    I.mvs_geom = cfg.mvs_detect_check && !(pe0 == 0 || a_end == 0 || pe0 < a_end || pe0 - a_end <= 2) &&
                 !(I.size < a_end + cfg.median_shift_window);
    I.win_var = !(pe0 - a_end <= cfg.pA_var_window + 2);
    I.win_mean = !(pe0 - a_end <= cfg.pA_mean_window + 2);
    I.smed_var = 0.f; I.smed_mean = 0.f;
    if (I.mvs_geom && (I.win_var || I.win_mean)) {
        const long long po = A.pre_off ? A.pre_off[r] : -1;
        if (!(po >= 0 && A.pre_meta[2 * r] == a_end && A.pre_meta[2 * r + 1] == pe0)) return false;
        I.smed_var = A.series_med[2 * r];
        I.smed_mean = A.series_med[2 * r + 1];
    }
    return true;
}

// the sample ranges whose order statistics the checks read: the adapter from 0 and from behind the last open pore, the
// local-range window of real_range_check (p15, p85), poly(A) from topk[0] (median; the MVS check's p15, p85), the MVS
// windows after / before adapter_end, the rest from polya_end, the median-shift windows after / before adapter_end.
// The MADs are those of A0, A1, P and R.
enum { VC_A0, VC_A1, VC_L15, VC_L85, VC_P, VC_P15, VC_P85, VC_AF, VC_BF, VC_R, VC_MA, VC_MB, VC_NQ };

struct VcGeom {
    int n_open, op_last;       // find_open_pores on the adapter: positions reported, the last one
    int ra, rlen;              // real_range_check window [a_start, a_end) (clipped)
    bool rr_geom;              // ... long enough for its two means
    int qa[VC_NQ], qb[VC_NQ];  // range q = samples [qa, qb) (clipped; empty: not wanted)
};

__device__ __forceinline__ VcGeom vc_geometry(const adb_config &cfg, const VcIn &I, int n_open, int op_last) {
    VcGeom G;
    G.n_open = n_open; G.op_last = op_last;
    const int a_end = I.a_end, pe_best = I.pe_best, size = I.size, msw = cfg.median_shift_window;
    const bool haveA = a_end != 0;
    const int a_start1 = (n_open > 0) ? op_last : 0;
    int ra = a_start1, rb = a_end;
    clip_seg(ra, rb, size);
    G.ra = ra; G.rlen = rb - ra;
    G.rr_geom = haveA && cfg.real_signal_check && G.rlen >= 2 * cfg.mean_window;
    const int lrw = min(cfg.max_obs_local_range, G.rlen);
    int pa_ = a_end, pb_ = I.pe0;
    clip_seg(pa_, pb_, size);
    const bool mvs_geom = I.mvs_geom, ms_geom = cfg.detect_med_shift && haveA;
#pragma unroll
    for (int q = 0; q < VC_NQ; q++) { G.qa[q] = 0; G.qb[q] = 0; }
    if (haveA) { G.qa[VC_A0] = 0; G.qb[VC_A0] = a_end; }
    if (haveA && a_start1 != 0) { G.qa[VC_A1] = a_start1; G.qb[VC_A1] = a_end; }
    if (G.rr_geom) { G.qa[VC_L15] = G.qa[VC_L85] = rb - lrw; G.qb[VC_L15] = G.qb[VC_L85] = rb; }
    if (mvs_geom || pe_best > a_end) { G.qa[VC_P] = a_end; G.qb[VC_P] = pe_best; }
    if (mvs_geom && pb_ > pa_) { G.qa[VC_P15] = G.qa[VC_P85] = a_end; G.qb[VC_P15] = G.qb[VC_P85] = I.pe0; }
    if (mvs_geom) {
        G.qa[VC_AF] = a_end; G.qb[VC_AF] = min(a_end + msw, size);
        G.qa[VC_BF] = max(a_end - msw, 0); G.qb[VC_BF] = a_end;
    }
    if (size > pe_best) { G.qa[VC_R] = pe_best; G.qb[VC_R] = size; }
    if (ms_geom) {
        G.qa[VC_MA] = a_end; G.qb[VC_MA] = min(a_end + cfg.med_shift_window, I.full_len);
        G.qa[VC_MB] = max(a_end - cfg.med_shift_window, 0); G.qb[VC_MB] = a_end;
    }
#pragma unroll
    for (int q = 0; q < VC_NQ; q++) clip_seg(G.qa[q], G.qb[q], size);
    return G;
}

__device__ __forceinline__ bool vc_is_pct(int q) { return q == VC_L15 || q == VC_L85 || q == VC_P15 || q == VC_P85; }

// np.percentile(method="linear") virtual index of a percentile range of n samples
__device__ __forceinline__ double vc_vindex(int q, int n) {
    return __dmul_rn((double)(n - 1), (q == VC_L15 || q == VC_P15) ? 0.15 : 0.85);
}

// rank k of the order statistic range q asks for (n > 0 samples), and whether numpy also needs rank k + 1
__device__ __forceinline__ int vc_rank(int q, int n, bool &two) {
    if (vc_is_pct(q)) {
        const int k = (int)floor(vc_vindex(q, n));
        two = min(k + 1, n - 1) != k;
        return k;
    }
    two = (n & 1) == 0;
    return (n - 1) / 2;
}

// what an order-statistic engine hands over to the checks (kept in shared memory by the kernels)
struct VcStats {
    int n[VC_NQ];              // samples of range q (0: not wanted)
    int c0[VC_NQ], c1[VC_NQ];  // codes at the ranks k and k + 1 of vc_rank (c1 = c0 when only one is needed)
    float mad[4];              // MADs of A0, A1, P, R
    float rm0, rm1;            // real_range_check: means of the first / last mean_window samples
    float small_mean, small_var;  // np.mean / np.var of the short poly(A) segment (when no moving window fits)
};

// small_mean / small_var of st when the checks need them: the short poly(A) segment [a_end, topk[0]) of the window w
// (at most pA_var_window + 2 samples).  One thread.
__device__ __forceinline__ void vc_small_mean_var(const VcIn &I, const int16_t *w, VcStats &st) {
    if (!I.mvs_geom || (I.win_var && I.win_mean)) return;
    int a = I.a_end, b = I.pe0;
    clip_seg(a, b, I.size);
    auto x = [&](int i) { return gsb_pa(w[a + i], I.coff, I.cscale); };
    st.small_mean = np_mean_f32(x, b - a);
    st.small_var = np_var_f32(x, b - a, st.small_mean);
}

// numpy median of range q
__device__ __forceinline__ float vc_median(const VcStats &st, int q, float coff, float cscale) {
    const int n = st.n[q];
    if (n <= 0) return CUDART_NAN_F;
    const float x0 = gsb_pa(st.c0[q], coff, cscale);
    if (n & 1) return x0;
    return __fdiv_rn(__fadd_rn(x0, gsb_pa(st.c1[q], coff, cscale)), 2.0f);
}

// p85 - p15 of the percentile ranges q15, q85
__device__ __forceinline__ double vc_local_range(const VcStats &st, int q15, int q85, float coff, float cscale) {
    if (st.n[q15] <= 0 || st.n[q85] <= 0) return CUDART_NAN;
    auto pct = [&](int q) {
        const double v = vc_vindex(q, st.n[q]);
        return np_lerp_f32(gsb_pa(st.c0[q], coff, cscale), gsb_pa(st.c1[q], coff, cscale), __dsub_rn(v, floor(v)));
    };
    const double p85 = pct(q85);
    return __dsub_rn(p85, pct(q15));
}

// the checks (combined.py:394-580); mode = ADB_METHOD_*
__device__ __forceinline__ VcOut vc_checks(const adb_config &cfg, const VcIn &I, const VcGeom &G, const VcStats &st, int mode,
                                           bool cand_followup) {
    VcOut o = vc_out(0);
    const int a_end = I.a_end, pe_best = I.pe_best;
    const float madA0 = st.mad[0];
    if (a_end == 0) { o.success = false; o.fail = ADB_FAIL_NO_ADAPTER; }
    if (o.success && (madA0 != 0.0f) && !in_range_d((double)madA0, cfg.adapter_mad_range)) { o.success = false; o.fail = ADB_FAIL_ADAPTER_MAD; }
    if (o.success && cfg.detect_open_pores) {
        o.n_open = G.n_open;
        o.valid |= ADB_V_OPEN_PORES;
        if (G.n_open > 0) {
            o.a_start = G.op_last;
            if (a_end - o.a_start < cfg.min_obs_adapter) { o.success = false; o.fail = ADB_FAIL_OPEN_PORE; }
        }
    }
    if (o.success && cfg.real_signal_check) {
        if (G.rlen < 2 * cfg.mean_window) {
            o.success = false; o.fail = ADB_FAIL_REAL_RANGE;
        } else {
            o.real[0] = (double)st.rm0; o.real[1] = (double)st.rm1;
            o.valid |= ADB_V_REAL_MEANS;
            if (in_range_d((double)st.rm0, cfg.mean_start_range) && in_range_d((double)st.rm1, cfg.mean_end_range)) {
                const double lr = vc_local_range(st, VC_L15, VC_L85, I.coff, I.cscale);
                o.real[2] = lr;
                o.valid |= ADB_V_REAL_RANGE;
                if (!in_range_d(lr, cfg.local_range)) { o.success = false; o.fail = ADB_FAIL_REAL_RANGE; }
            } else {
                o.success = false; o.fail = ADB_FAIL_REAL_RANGE;
            }
        }
    }
    bool need_mvs = false;
    double mr[2];
    if (o.success && cfg.mvs_detect_check) {
        if (pe_best == 0) {
            o.success = false; o.fail = ADB_FAIL_NO_POLYA;
        } else {
            if (!vc_pa_mean_bounds(cfg, vc_median(st, VC_A0, I.coff, I.cscale), mr)) { o.exception = true; o.fail = ADB_FAIL_EXC_PA_MEAN_RANGE; }
            else if (I.n_topk < 0) { o.exception = true; o.fail = ADB_FAIL_EXC_TOPK_NONE; }
            need_mvs = !o.exception && I.n_topk >= 1 && I.pe0 != 0;
        }
    }
    if (need_mvs) {
        // first candidate (mvs.py:45-158)
        o.valid |= ADB_V_MVS;
        bool ok = false;
        if (I.mvs_geom) {
            o.mvs[0] = (double)(I.win_mean ? I.smed_mean : st.small_mean);
            o.mvs[1] = (double)(I.win_var ? I.smed_var : st.small_var);
            o.mvs[2] = (double)vc_median(st, VC_P, I.coff, I.cscale);
            o.mvs[3] = vc_local_range(st, VC_P15, VC_P85, I.coff, I.cscale);
            o.mvs[4] = (double)__fsub_rn(vc_median(st, VC_AF, I.coff, I.cscale), vc_median(st, VC_BF, I.coff, I.cscale));
            const int mask = vc_mvs_mask(cfg, o.mvs, mr);
            ok = (mask == 0);
            if (!ok) { o.success = false; vc_mvs_fail(o.mvs[0], mask, o.fail, o.fail_mask); }
        } else {
            o.success = false; o.fail = ADB_FAIL_MVS_NOT_ENOUGH; o.fail_mask = 0;
        }
        if (!ok && I.topk1 != 0) {
            // the reference goes on to the next candidates (combined.py:464-515): their moving statistics are
            // prefixes of one more series pass, so validate_cand_kernel finishes the read from this record
            if (cand_followup) o.followup = true; else o.defer = true;
        }
    }
    if (!o.exception && o.success && cfg.detect_med_shift) {
        o.med_shift = (double)__fsub_rn(vc_median(st, VC_MA, I.coff, I.cscale), vc_median(st, VC_MB, I.coff, I.cscale));
        o.valid |= ADB_V_MED_SHIFT;
        if (!in_range_d(o.med_shift, cfg.med_shift_range)) { o.success = false; o.fail = ADB_FAIL_MED_SHIFT; }
    }
    if (mode == ADB_METHOD_CNN && cfg.fallback_to_llr_short_reads && !o.exception && !o.success && a_end > 0 && pe_best > 0 &&
        pe_best - a_end > 1000 && I.full_len < 2 * cfg.max_obs_adapter)
        o.defer = true;  // "hail mary" LLR fallback (combined.py:251-301) lives in validate_kernel
    return o;
}

// partition p of the record (0 adapter, 1 poly(A), 2 the rest): samples [a, b); false when empty
__device__ __forceinline__ bool vc_partition(const VcIn &I, const VcOut &o, int p, int &a, int &b) {
    a = (p == 0) ? o.a_start : (p == 1) ? I.a_end : I.pe_best;
    b = (p == 0) ? I.a_end : (p == 1) ? I.pe_best : I.size;
    return b > a;
}

// mean / population std of the pA values of n samples from the exact sums of their codes s1 = sum c, s2 = sum c^2
// (signal_partitions.py:91-92; numpy sums float32 pairwise -- the contract for these statistics is 1e-5 relative)
__device__ __forceinline__ void vc_mean_std(long long s1, long long s2, int n, float coff, float cscale, double &mean, double &std) {
    const double mk = (double)s1 / n;
    double vk = (double)s2 / n - mk * mk;
    if (vk < 0) vk = 0;
    mean = (double)(float)((mk + (double)coff) * (double)cscale);
    std = (double)(float)(sqrt(vk) * fabs((double)cscale));
}

// the record of a read the checks have settled (not deferred), with the partitions' mean / std.  One thread.
__device__ __forceinline__ void vc_write_spec_record(adb_record *rec, const VcIn &I, const VcStats &st, VcOut o, const double pmean[3],
                                                     const double pstd[3]) {
    if (o.exception) { vc_write_exception(rec, o.fail, I.full_len, I.size); return; }
    double tab[3][4];
    for (int p = 0; p < 3; p++) for (int q = 0; q < 4; q++) tab[p][q] = 0.0;
    const int medq[3] = {o.a_start == 0 ? VC_A0 : VC_A1, VC_P, VC_R};
    const float mad[3] = {o.a_start == 0 ? st.mad[0] : st.mad[1], st.mad[2], st.mad[3]};
    const uint32_t bit[3] = {ADB_V_ADAPTER_STATS, ADB_V_POLYA_STATS, ADB_V_RNA_STATS};
    for (int p = 0; p < 3; p++) {
        int a, b;
        if (!vc_partition(I, o, p, a, b)) continue;
        tab[p][0] = pmean[p]; tab[p][1] = pstd[p]; tab[p][2] = (double)vc_median(st, medq[p], I.coff, I.cscale); tab[p][3] = (double)mad[p];
        o.valid |= bit[p];
    }
    vc_write_record(rec, o, tab, I.full_len, I.size, I.a_end, I.pe_best, I.a_end, I.pe_best, 0, I.n_topk, I.g + 1);
    if (o.followup) *reinterpret_cast<float *>(rec->_reserved) = vc_median(st, VC_A0, I.coff, I.cscale);  // scales the mean range of the later candidates
}
