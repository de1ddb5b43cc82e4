// Per-read kernels (one CTA per read, persistent over the reads of a call).
//
//   llr_primary_kernel   LLR primary boundaries (combined_detect_llr2 up to the Boundaries object, combined.py:128-211):
//                        clip / normalise with the minibatch-global med/MAD -> float32 mean-pool downscale in numpy's
//                        pairwise order -> sequential float64 prefix sums -> adapter LLR trace -> first surviving peak
//                        (+ plateau / split fixes) -> poly(A) LLR trace -> spike rule.  Small shared-memory footprint
//                        (3 x nds doubles); one WARP per read (CTAs of 32 threads), so that the strictly sequential
//                        pieces (prefix sums, peak walks) of one read overlap the parallel pieces of the others.
//   validate_kernel      validate_boundaries + partition statistics (combined.py:358-631) for boundaries taken from
//                        a device array (LLR / CNN / start-peak primaries alike), plus the CNN path's "hail mary"
//                        LLR fallback (combined.py:251-301).  The read's preload window is staged ONCE in shared
//                        memory by the TMA bulk engine (cp.async.bulk + mbarrier) and every order statistic, moving
//                        statistic and sum is computed from there.  Windows too long for that (win_bytes == 0) are
//                        read straight from global memory; shared memory then holds only the scratch, and the
//                        hail-mary trace keeps its prefix sums in global memory.
//
// Primary boundaries travel between the two as int[n_reads][stride]: adapter_end, polya_end, top-k...,
// with n_topk == -1 encoded as polya_end_topk = None.
#pragma once
#include "adb_common.cuh"
#include "adb_global.cuh"
#include "adb_llr.cuh"
#include "adb_select.cuh"
#include "adb_validate.cuh"
#include "adb_vfast.cuh"

#define ADB_TRACE_THREADS 64    // two warps per read and up to 16 reads in flight per SM: the serial pieces of one read
                                // (prefix chains, peak walks on warp 0) run under the parallel pieces of the others
#define ADB_VAL_THREADS 256

// float32 mean of one downscale block in numpy's pairwise order (SURVEY a2).  f(k) = k-th sample of the block.
template <class F>
__device__ __forceinline__ float block_mean_f32(F f, int factor) {
    return __fdiv_rn(np_sum_f32_leaf(f, factor), (float)factor);
}

// block mean with all loads issued first (compile-time factor): one memory latency per block instead of `factor`
template <int FACT, class F>
__device__ __forceinline__ float block_mean_f32_fixed(F f) {
    float v[FACT];
#pragma unroll
    for (int k = 0; k < FACT; k++) v[k] = f(k);
    return __fdiv_rn(np_sum_f32_leaf([&](int k) { return v[k]; }, FACT), (float)FACT);
}

struct TraceScratch {
    double *trace, *c, *c2;
    PeakScratch PS;
    int *itmp;
    double *dtmp;
};

// c_ext == true: the two prefix-sum arrays live in global memory (llr_primary_kernel: a third of the shared-memory
// footprint per read, so that twice as many reads are in flight per SM)
__host__ __device__ inline size_t trace_smem_bytes(int nds_max, int peak_cap, bool c_ext = false) {
    return (size_t)nds_max * (c_ext ? 8 : 24) + (((size_t)peak_cap * 6 + 15) & ~(size_t)15) + 128;
}

__device__ __forceinline__ TraceScratch trace_scratch_from(unsigned char *base, int nds_max, int peak_cap, double *c_ext = nullptr) {
    TraceScratch T;
    T.trace = (double *)base;
    T.c = c_ext ? c_ext : T.trace + nds_max;
    T.c2 = T.c + nds_max;
    unsigned char *after = c_ext ? (unsigned char *)(T.trace + nds_max) : (unsigned char *)(T.c2 + nds_max);
    T.PS.cap = peak_cap;
    T.PS.pk = (unsigned short *)after;
    T.PS.stack = T.PS.pk + peak_cap;
    T.PS.status = (unsigned char *)(T.PS.stack + peak_cap);
    T.PS.flags = T.PS.status + peak_cap;
    unsigned char *small = after + (((size_t)peak_cap * 6 + 15) & ~(size_t)15);
    T.itmp = (int *)small;            // 8 ints
    T.dtmp = (double *)(small + 64);  // 8 doubles
    return T;
}

// LLR boundaries on the downscaled, normalised row ds[0..nds) (float32, aliasing T.trace).
// Outputs (uniform): ae_ds (-1: no candidate), pe_ds (0: none).  CTA-wide.
__device__ void llr_boundaries_cta(const float *ds, int nds, const TraceScratch &T, const adb_config &cfg,
                                   bool adapter_stage, int &ae_ds, int &pe_ds) {
    double *trace = T.trace, *c = T.c, *c2 = T.c2;
    // sequential float64 prefix sums (_c_llr.pyx:216-217): the two chains run in lockstep on lanes 0 (x) and 1 (x*x)
    // of the first warp; loads are hoisted four elements ahead so that only the dependent adds remain on the chain
    if (threadIdx.x < 2) {
        const bool sq = threadIdx.x == 1;
        double *dst = sq ? c2 : c;
        double s = 0.0;
        int i = 0;
        for (; i + 4 <= nds; i += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(ds + i);  // ds is 16-byte aligned (start of the trace buffer)
            double x0 = (double)v.x, x1 = (double)v.y, x2 = (double)v.z, x3 = (double)v.w;
            if (sq) { x0 = __dmul_rn(x0, x0); x1 = __dmul_rn(x1, x1); x2 = __dmul_rn(x2, x2); x3 = __dmul_rn(x3, x3); }
            s = __dadd_rn(s, x0); dst[i] = s;
            s = __dadd_rn(s, x1); dst[i + 1] = s;
            s = __dadd_rn(s, x2); dst[i + 2] = s;
            s = __dadd_rn(s, x3); dst[i + 3] = s;
        }
        for (; i < nds; i++) {
            double x = (double)ds[i];
            if (sq) x = __dmul_rn(x, x);
            s = __dadd_rn(s, x);
            dst[i] = s;
        }
    }
    __syncthreads();
    ae_ds = 0;
    pe_ds = 0;
    if (adapter_stage) {
        // adapter trace: start 0, end nds-1, head 5, tail 5 (combined.py:155-170)
        cta_llr_gains(c, c2, nds, 0, nds - 1, 5, 5, 1, trace);
        int s0, e0;
        cta_trace_support(trace, nds, s0, e0, T.itmp);
        if (threadIdx.x < 32) { const double sd = warp_nanstd(trace, s0, e0); if (threadIdx.x == 0) T.dtmp[0] = sd; }
        __syncthreads();
        const double pmin = __dmul_rn(cfg.adapter_peak_prominence, T.dtmp[0]);
        const double wmin = (double)(cfg.adapter_peak_width / cfg.downscale_factor);
        ae_ds = cta_adapter_end(trace, nds, s0, e0, pmin, wmin, cfg.adapter_peak_rel_height, T.PS, T.itmp + 4);
        if (ae_ds < 0) return;
        // poly(A) trace: start = adapter_end, head 1, tail 1, same prefix sums (combined.py:189-204)
        cta_llr_gains(c, c2, nds, ae_ds, nds - 1, 1, 1, 1, trace);
    } else {
        // hail-mary variant: a single trace (head 5, tail 5) feeds the spike rule directly (combined.py:277-292)
        cta_llr_gains(c, c2, nds, 0, nds - 1, 5, 5, 1, trace);
    }
    pe_ds = cta_polya_end(trace, nds, T.PS, T.itmp + 4);
}

// normalised, clipped sample j of the read (normalize.py:25-28,61-63), float32 steps
__device__ __forceinline__ float norm_sample(const ReadSrc &src, int j, float lo, float hi, float med, float mad) {
    float v = src.pa(j);
    v = (v < lo) ? lo : ((v > hi) ? hi : v);  // np.clip keeps NaN
    return __fdiv_rn(__fsub_rn(v, med), mad);
}

struct PrimaryArgs {
    BatchDev B;
    const GselState *gstates;
    int nds_max, peak_cap;
    int *given;        // out: [n_reads][2]
    int *ntopk;        // out: [n_reads] (-1: None, 1: one candidate)
    int *batch_status;
    double *cc;        // [gridDim.x][2][nds_max] prefix sums of the read a CTA works on (global memory, L1 / L2 resident)
};

__global__ void __launch_bounds__(ADB_TRACE_THREADS, 16) llr_primary_kernel(PrimaryArgs A, adb_config cfg) {
    extern __shared__ __align__(16) unsigned char smem[];
    const TraceScratch T = trace_scratch_from(smem, A.nds_max, A.peak_cap, A.cc + (size_t)blockIdx.x * 2 * A.nds_max);
    float *ds = (float *)T.trace;
    // While the downscaled row (float32) occupies the first half of the trace buffer, its second half holds a per-read
    // table of the normalised values: for int16 reads the clipped, normalised sample is a function of the ADC code
    // alone and the clip interval spans a few hundred codes, so the IEEE division runs once per code of that interval
    // instead of once per raw sample (same operations on the same operands: bit-identical).
    float *lut = ds + A.nds_max;
    // the reference slices batch[:, :max_obs_trace] (combined.py:128-136): a matrix narrower than that keeps its own width
    const int Tm = min(cfg.max_obs_trace, A.B.m), A0 = cfg.min_obs_adapter, f = cfg.downscale_factor;
    for (int r = blockIdx.x; r < A.B.n_reads; r += gridDim.x) {
        const int mb = r / A.B.batch_size;
        __syncthreads();
        if (threadIdx.x == 0) { A.given[2 * r] = 0; A.given[2 * r + 1] = 0; A.ntopk[r] = -1; }
        const GselState gs = A.gstates[mb];
        if (gs.status != ADB_OK) continue;  // minibatch lost (host raises)
        const ReadSrc src = make_src(A.B, r);
        // pull the trace window of the NEXT read of this warp into L2 while this one is processed (one warp per read
        // at low occupancy: the loads of the downscale step would otherwise wait on HBM)
        if (r + (int)gridDim.x < A.B.n_reads && A.B.sig_type == ADB_SIG_I16) {
            const int rn = r + gridDim.x;
            const int64_t o0 = A.B.offsets[rn], o1 = A.B.offsets[rn + 1];
            const int nn = (int)min((int64_t)Tm, o1 - o0);
            const char *p = (const char *)((const int16_t *)A.B.signal + o0 + A0);
            const int bytes = max(nn - A0, 0) * 2;
            for (int b = threadIdx.x * 128; b < bytes; b += blockDim.x * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p + b));
        }
        // number of non-NaN downscaled bins (combined.py:133-154)
        int nds;
        {
            const int L = min(src.n, Tm) - A0;
            if (src.n >= Tm) nds = (Tm - A0 + f - 1) / f;
            else nds = (L > 0) ? L / f : 0;
            if (Tm - A0 <= 0) nds = 0;
        }
        if (nds <= 0) {
            if (threadIdx.x == 0) atomicMin(&A.batch_status[mb], (int)ADB_ERR_EMPTY_TRACE);
            continue;
        }
        const float med = gs.med, mad = gs.mad;
        const float lo = (float)((double)med - (double)mad * cfg.sig_norm_outlier_thresh);
        const float hi = (float)((double)med + (double)mad * cfg.sig_norm_outlier_thresh);
        // all blocks but a zero-padded ragged last one are complete
        const int nfull = (Tm - A0) / f;
        // table of the normalised values over the codes of the clip interval (+ 2 codes on either side): everything
        // below its first code clips to `lo`, everything above its last code to `hi` -- verified, else computed directly
        int c_base = 0, c_top = -1;
        if (src.i16 && src.cscale > 0.0f) {
            const float fb = floorf(lo / src.cscale - src.coff) - 2.0f, ft = ceilf(hi / src.cscale - src.coff) + 2.0f;
            if (fb >= -40000.0f && ft <= 40000.0f && ft >= fb) {
                c_base = max((int)fb, -32768);
                c_top = min((int)ft, 32767);
                const bool ok = (c_top - c_base + 1 <= A.nds_max) && c_top >= c_base &&
                                (c_base == -32768 || __fmul_rn(__fadd_rn((float)c_base, src.coff), src.cscale) <= lo) &&
                                (c_top == 32767 || __fmul_rn(__fadd_rn((float)c_top, src.coff), src.cscale) >= hi);
                if (!ok) c_top = c_base - 1;
            }
        }
        const bool use_lut = c_top >= c_base;  // uniform: derived from per-read constants only
        if (use_lut) {
            for (int e = threadIdx.x; e <= c_top - c_base; e += blockDim.x) {
                float v = __fmul_rn(__fadd_rn((float)(c_base + e), src.coff), src.cscale);
                v = (v < lo) ? lo : ((v > hi) ? hi : v);
                lut[e] = __fdiv_rn(__fsub_rn(v, med), mad);
            }
            __syncthreads();
            const int top_e = c_top - c_base;
            const int16_t *codes = src.i16;
            auto look = [&](int j) { return lut[min(max((int)codes[j] - c_base, 0), top_e)]; };
            for (int b = threadIdx.x; b < nds; b += blockDim.x) {
                const int j0 = A0 + b * f;
                float v;
                if (b < nfull && f == 20) v = block_mean_f32_fixed<20>([&](int k) { return look(j0 + k); });
                else if (b < nfull && f == 10) v = block_mean_f32_fixed<10>([&](int k) { return look(j0 + k); });
                else v = block_mean_f32([&](int k) { const int j = j0 + k; return (j >= Tm) ? 0.0f : look(j); }, f);
                ds[b] = v;
            }
        } else {
            for (int b = threadIdx.x; b < nds; b += blockDim.x) {
                const int j0 = A0 + b * f;
                float v;
                if (b < nfull && f == 20) v = block_mean_f32_fixed<20>([&](int k) { return norm_sample(src, j0 + k, lo, hi, med, mad); });
                else if (b < nfull && f == 10) v = block_mean_f32_fixed<10>([&](int k) { return norm_sample(src, j0 + k, lo, hi, med, mad); });
                else
                    v = block_mean_f32(
                        [&](int k) {
                            const int j = j0 + k;
                            return (j >= Tm) ? 0.0f : norm_sample(src, j, lo, hi, med, mad);  // np.pad zero padding
                        },
                        f);
                ds[b] = v;
            }
        }
        __syncthreads();
        int ae_ds, pe_ds;
        llr_boundaries_cta(ds, nds, T, cfg, true, ae_ds, pe_ds);
        if (threadIdx.x == 0) {
            int ae = 0, pe = 0, nt = -1;
            if (ae_ds > 0) ae = ae_ds * f + A0;
            if (ae_ds >= 0 && pe_ds > 0) { pe = pe_ds * f + A0; nt = 1; }
            A.given[2 * r] = ae;
            A.given[2 * r + 1] = pe;
            A.ntopk[r] = nt;
        }
    }
}

struct ValidateArgs {
    BatchDev B;
    const int *given;     // [n_reads][given_stride] = adapter_end, polya_end(= topk[0]), topk[1..]
    int given_stride;
    int given_ntopk;      // entries per read when ntopk_per_read == nullptr (-1: None)
    const int *ntopk_per_read;  // optional per-read override (LLR: -1 / 1)
    int mode;             // ADB_METHOD_*
    int win_bytes;        // capacity of the staged window (bytes); 0: the window is read from global memory
    int nds_max, peak_cap;// hail-mary trace buffers (CNN mode only; 0 otherwise)
    double *hm_cc;        // [gridDim.x][2][nds_max] hail-mary prefix sums in global memory (nullptr: in shared memory)
    adb_record *out;
    float *series;        // [gridDim.x][2][m]
    const int *batch_status;
    const float *pre_var, *pre_mean;  // compact pools of precomputed moving statistics (mvs_series_kernel)
    const long long *pre_off;         // [n_reads] row offset into the pools, -1: none
    const int *pre_meta;              // [n_reads][2] = (adapter_end, polya_end) of the row
    const unsigned char *done;        // optional [n_reads]: 1 = already written by validate_fast_kernel
    // optional compact list of the reads still to do (mvs_pending_kernel) + a work counter: CTAs then take the next
    // read of the list dynamically -- the handed-over reads are few and of very uneven cost (several poly(A)
    // candidates, hail-mary trace), a static stride would leave most CTAs idle behind the unlucky ones
    const int *pending, *n_pending;
    int *work_counter;
};

// shared memory of validate_kernel: [window (+48)][scratch: select histogram | hail-mary trace buffers][small].
// win_bytes == 0: no staged window; c_ext: the trace's prefix sums live in global memory.
__host__ __device__ inline size_t validate_win_cap(int win_bytes) {
    return win_bytes > 0 ? (((size_t)win_bytes + 48 + 15) & ~(size_t)15) : 0;
}
__host__ __device__ inline size_t validate_scratch_bytes(int nds_max, int peak_cap, bool c_ext) {
    size_t scratch = ADB_SEL_SMEM_BYTES + 64;
    size_t tr = nds_max > 0 ? trace_smem_bytes(nds_max, peak_cap, c_ext) : 0;
    if (tr > scratch) scratch = tr;
    return (scratch + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t validate_smem_bytes(int win_bytes, int nds_max, int peak_cap, bool c_ext = false) {
    return validate_win_cap(win_bytes) + validate_scratch_bytes(nds_max, peak_cap, c_ext) + 256;
}

// A.win_bytes > 0: the read's window is copied to shared memory first; 0: every reader works on the read in global
// memory (the same plain loads; the staged copy keeps the source's 16-byte phase and nobody reads past the read's
// samples, so the readers see the same data either way).  One kernel for both: a second instantiation would give the
// large device functions two call sites and change how they are inlined.
__global__ void __launch_bounds__(ADB_VAL_THREADS, 3) validate_kernel(ValidateArgs A, adb_config cfg) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *winbuf = smem;
    unsigned char *scratch = smem + validate_win_cap(A.win_bytes);
    const bool c_ext = A.hm_cc != nullptr;
    const size_t scratch_sz = validate_scratch_bytes(A.nds_max, A.peak_cap, c_ext);
    unsigned char *small = scratch + scratch_sz;
    uint32_t *kbuf = (uint32_t *)small;          // 8 words
    int *itmp = (int *)(small + 32);             // 8 ints
    double *dtmp = (double *)(small + 64);       // 8 doubles
    int *topk_sh = (int *)(small + 128);         // ADB_MAX_CAND ints
    uint64_t *bar = (uint64_t *)(small + 192);

    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    uint32_t phase = 0;

    ValCtx C;
    C.cfg = &cfg;
    C.S = sel_scratch_from(scratch);
    C.kbuf = kbuf;
    C.itmp = itmp;
    C.dtmp = dtmp;
    C.series_a = A.series + (size_t)blockIdx.x * 2 * A.B.m;
    C.series_b = C.series_a + A.B.m;

    int *next_sh = (int *)(small + 200);
    for (int step = blockIdx.x;; step += gridDim.x) {
        int r;
        if (A.pending) {
            __syncthreads();
            if (threadIdx.x == 0) *next_sh = atomicAdd(A.work_counter, 1);
            __syncthreads();
            const int idx = *next_sh;
            if (idx >= *A.n_pending) break;
            r = A.pending[idx];
        } else {
            r = step;
            if (r >= A.B.n_reads) break;
        }
        const int mb = r / A.B.batch_size;
        adb_record *rec = A.out + r;
        __syncthreads();
        if (A.done && A.done[r]) continue;
        {
            const long long po = A.pre_off ? A.pre_off[r] : -1;
            C.pre_var = (po >= 0) ? A.pre_var + po : nullptr;
            C.pre_mean = (po >= 0) ? A.pre_mean + po : nullptr;
            C.pre_ae = (po >= 0) ? A.pre_meta[2 * r] : -1;
            C.pre_pe = (po >= 0) ? A.pre_meta[2 * r + 1] : -1;
        }
        // zero the record (so unset groups read as zeros) -- 512 B = 128 words
        for (int w = threadIdx.x; w < (int)(sizeof(adb_record) / 4); w += blockDim.x) ((uint32_t *)rec)[w] = 0;
        if (A.batch_status[mb] != ADB_OK) continue;  // minibatch lost (host raises)
        const ReadSrc gsrc = make_src(A.B, r);
        const int full_len = A.B.full_lens[r];
        // ---- stage the preload window in shared memory (TMA bulk copy) ----
        ReadSrc src = gsrc;
        if (A.win_bytes > 0) {
            const int esz = gsrc.f32 ? 4 : 2;
            const unsigned char *g = gsrc.f32 ? (const unsigned char *)gsrc.f32 : (const unsigned char *)gsrc.i16;
            unsigned char *w = cta_stage_window(winbuf, g, gsrc.n * esz, bar, phase);
            if (gsrc.f32) src.f32 = (const float *)w; else src.i16 = (const int16_t *)w;
        }
        C.src = src;
        C.int_keys = (src.i16 != nullptr) && (src.cscale > 0.0f);

        PrimaryBounds PB;
        PB.adapter_start = 0;
        PB.topk = topk_sh;
        {
            const int *g = A.given + (size_t)r * A.given_stride;
            PB.adapter_end = g[0];
            PB.polya_end = g[1];
            PB.n_topk = A.ntopk_per_read ? A.ntopk_per_read[r] : A.given_ntopk;
            if (threadIdx.x < ADB_MAX_CAND) topk_sh[threadIdx.x] = (threadIdx.x < PB.n_topk) ? g[1 + threadIdx.x] : 0;
        }
        __syncthreads();

        val_window_bounds(C);
        validate_boundaries_cta(C, PB, full_len, rec);

        if (A.mode == ADB_METHOD_CNN && A.nds_max > 0) {
            // "hail mary" LLR fallback for short reads (combined.py:251-301)
            __syncthreads();
            const bool failed = (rec->success == 0) && (rec->valid & ADB_V_FIELDS);
            const int ae = PB.adapter_end, pe = PB.polya_end;
            if (failed && ae > 0 && pe > 0 && pe - ae > 1000 && full_len < 2 * cfg.max_obs_adapter &&
                cfg.fallback_to_llr_short_reads) {
                // per-read normalisation over signal[:min(max_obs_trace, full_len)] (NaN padding dropped)
                const int nn = min(min(cfg.max_obs_trace, full_len), A.B.m);
                const int nvalid = min(nn, src.n);
                const SegStats N0 = seg_stats(C, 0, nvalid, SS_MED | SS_MAD);
                const float med = N0.med, mad = N0.mad;
                if (nvalid > 0 && mad == 0.0f) {
                    // normalize_signal raises ValueError("MAD normalization failed: scale is 0") inside the try
                    __syncthreads();
                    if (threadIdx.x == 0) { rec->valid = 0; rec->success = 0; rec->fail_code = ADB_FAIL_EXC_MAD_ZERO; }
                    continue;
                }
                const float lo = (float)((double)med - (double)mad * cfg.sig_norm_outlier_thresh);
                const float hi = (float)((double)med + (double)mad * cfg.sig_norm_outlier_thresh);
                const int f = cfg.downscale_factor;
                // norm_signal[ae:pe] (clipped to nn), zero padded to a multiple of f, NaN where the read has ended
                const int sa = min(ae, nn), sb = min(pe, nn);
                const int seglen = sb - sa;
                const int nblk = (seglen + f - 1) / f;
                // leading NaN-free blocks: a block is NaN iff it reaches past the read's last sample
                int nds;
                if (sb <= nvalid) nds = nblk;
                else nds = (nvalid > sa) ? (nvalid - sa) / f : 0;
                if (nds > A.nds_max) nds = A.nds_max;
                if (nds <= 0) {
                    __syncthreads();
                    if (threadIdx.x == 0) { rec->valid = 0; rec->success = 0; rec->fail_code = ADB_FAIL_EXC_EMPTY_TRACE; }
                    continue;
                }
                __syncthreads();
                const TraceScratch T = trace_scratch_from(scratch, A.nds_max, A.peak_cap,
                                                          c_ext ? A.hm_cc + (size_t)blockIdx.x * 2 * A.nds_max : nullptr);
                float *ds = (float *)T.trace;
                for (int b = threadIdx.x; b < nds; b += blockDim.x) {
                    const int j0 = sa + b * f;
                    ds[b] = block_mean_f32(
                        [&](int k) {
                            const int j = j0 + k;
                            return (j >= sb) ? 0.0f : norm_sample(src, j, lo, hi, med, mad);
                        },
                        f);
                }
                __syncthreads();
                int ae_ds, pe_ds;
                llr_boundaries_cta(ds, nds, T, cfg, false, ae_ds, pe_ds);
                if (pe_ds > 0) {
                    PB.polya_end = pe_ds * f + ae;
                    PB.n_topk = 1;
                    __syncthreads();
                    if (threadIdx.x == 0) topk_sh[0] = PB.polya_end;
                    for (int w = threadIdx.x; w < (int)(sizeof(adb_record) / 4); w += blockDim.x) ((uint32_t *)rec)[w] = 0;
                    __syncthreads();
                    validate_boundaries_cta(C, PB, full_len, rec);
                }
            }
        }
    }
}
