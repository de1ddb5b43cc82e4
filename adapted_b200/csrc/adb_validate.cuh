// validate_boundaries + per-segment statistics, one CTA per read.
//
// Reference: adapted/detect/combined.py:358-631 with adapted/detect/anomalies.py:15-35 (open pores),
// adapted/detect/real_range.py:33-63, adapted/detect/mvs.py:45-158 (mean/var/median-shift check, bottleneck
// moving statistics restated from its move_template.c recurrences in float32), adapted/detect/utils.py:16-36,
// adapted/partition/signal_partitions.py:65-96.  Control flow follows SURVEY.md A.8 including the
// "success is never reset" behaviour of the top-k loop.
#pragma once
#include "adb_common.cuh"
#include "adb_select.cuh"
#include "adb_vcheck.cuh"

#define ADB_MAX_MOVE_WINDOW 4096   // bottleneck window sizes accepted (any value up to the segment length works)
#define ADB_MAX_MEAN_WINDOW 65536

struct ValCtx {
    ReadSrc src;         // the read's preload window: staged in shared memory, or the read in global memory
    const adb_config *cfg;
    SelScratch S;
    uint32_t *kbuf;      // shared: 4 keys + 4 ranks
    float *series_a;     // global scratch [m] (moving variance)  -- in-CTA fallback path
    float *series_b;     // global scratch [m] (moving mean)
    const float *pre_var;   // moving variance of candidate 0 precomputed by mvs_series_kernel (or nullptr)
    const float *pre_mean;  // moving mean of candidate 0
    int pre_ae, pre_pe;     // the (adapter_end, polya_end) pair the precomputed series belong to (-1: none)
    int *itmp;           // shared: 8 ints
    double *dtmp;        // shared: 8 doubles
    bool int_keys;       // raw ADC keys usable (i16 source, scale > 0)
    uint32_t wkmin, wkmax;  // key bounds of the whole window
    float wvmin, wvmax;     // value bounds of the whole window
};

// ---- keys of a pA segment ----------------------------------------------------------------------------------
struct PaKeys {
    ReadSrc s;
    int a;
    bool ik;
    __device__ __forceinline__ uint32_t operator()(int j) const {
        if (ik) return (uint32_t)((int)s.i16[a + j] + 32768);
        return f32_key(s.pa(a + j));
    }
};
struct PaVal {
    ReadSrc s;
    bool ik;
    __device__ __forceinline__ float operator()(uint32_t k) const {
        if (ik) return __fmul_rn(__fadd_rn((float)((int)k - 32768), s.coff), s.cscale);
        return key_f32(k);
    }
};
struct DevKeys {  // |x - med| in float32
    ReadSrc s;
    int a;
    float med;
    __device__ __forceinline__ uint32_t operator()(int j) const { return f32_key(fabsf(__fsub_rn(s.pa(a + j), med))); }
};
struct BufKeys {
    const float *p;
    __device__ __forceinline__ uint32_t operator()(int j) const { return f32_key(p[j]); }
};
struct KeyToF32 {
    __device__ __forceinline__ float operator()(uint32_t k) const { return key_f32(k); }
};

__device__ void val_window_bounds(ValCtx &C) {
    PaKeys K{C.src, 0, C.int_keys};
    PaVal V{C.src, C.int_keys};
    cta_key_minmax(K, C.src.n, C.wkmin, C.wkmax, C.S);
    if (C.src.n > 0) {
        C.wvmin = V(C.wkmin);
        C.wvmax = V(C.wkmax);
    } else {
        C.wvmin = C.wvmax = 0.f;
        C.wkmin = C.wkmax = 0;
    }
}

__device__ float seg_median(ValCtx &C, int a, int b) {
    clip_seg(a, b, C.src.n);
    PaKeys K{C.src, a, C.int_keys};
    PaVal V{C.src, C.int_keys};
    return cta_median_keys(K, V, b - a, C.wkmin, C.wkmax, C.S, C.kbuf);
}

// median(|x - med|) in float32 (combined.py:399-400, signal_partitions.py:94)
__device__ float seg_mad(ValCtx &C, int a, int b, float med) {
    clip_seg(a, b, C.src.n);
    if (b - a <= 0) return CUDART_NAN_F;
    if (!(med == med)) return CUDART_NAN_F;
    DevKeys K{C.src, a, med};
    float dmax = fmaxf(fabsf(__fsub_rn(C.wvmax, med)), fabsf(__fsub_rn(C.wvmin, med)));
    return cta_median_keys(K, KeyToF32(), b - a, f32_key(0.0f), f32_key(dmax), C.S, C.kbuf);
}

// np.subtract(*np.percentile(seg, (85, 15))) -> float64 (real_range.py:50-57, mvs.py:113-118)
__device__ double seg_local_range(ValCtx &C, int a, int b) {
    clip_seg(a, b, C.src.n);
    const int n = b - a;
    if (n <= 0) return CUDART_NAN;
    int *ranks = (int *)(C.kbuf + 4);
    // virtual indexes (n-1)*q in float64, q = 85/100, 15/100
    const double v85 = __dmul_rn((double)(n - 1), 0.85), v15 = __dmul_rn((double)(n - 1), 0.15);
    const int l85 = (int)floor(v85), l15 = (int)floor(v15);
    const int h85 = min(l85 + 1, n - 1), h15 = min(l15 + 1, n - 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        // ascending, possibly equal ranks: l15 <= h15 <= l85 <= h85
        ranks[0] = l15; ranks[1] = h15; ranks[2] = l85; ranks[3] = h85;
    }
    __syncthreads();
    PaKeys K{C.src, a, C.int_keys};
    PaVal V{C.src, C.int_keys};
    cta_select_ranks(K, n, C.wkmin, C.wkmax, ranks, 4, C.kbuf, C.S);
    const float a15 = V(C.kbuf[0]), b15 = V(C.kbuf[1]), a85 = V(C.kbuf[2]), b85 = V(C.kbuf[3]);
    const double p85 = np_lerp_f32(a85, b85, __dsub_rn(v85, (double)l85));
    const double p15 = np_lerp_f32(a15, b15, __dsub_rn(v15, (double)l15));
    __syncthreads();
    return __dsub_rn(p85, p15);
}

// ---- segment statistics from ONE histogram pass (int16 sources) -------------------------------------------------
// pA = (adc + offset) * scale is monotone in the ADC code for scale > 0, so order statistics can be taken in the
// integer domain and mapped back exactly.  A read spans 1-2 k distinct codes, so one shared-memory histogram over
// [wkmin, wkmax] holds a whole segment; after an in-place inclusive scan it answers, without touching the samples
// again:  median (two rank look-ups), p85 - p15 (four look-ups + numpy's float64 lerp), and the MAD -- the k-th
// smallest |pA(code) - med| found by counting, with two binary searches per occupied code, how many samples deviate
// less (deviations are monotone on either side of the median).  Sources that do not qualify (float32 input,
// non-positive scale, > ADB_SEL_NB codes) use the generic multi-level select above.
#define SS_MED 1
#define SS_MAD 2
#define SS_LR 4
struct SegStats {
    float med, mad;
    double lr;
};

__device__ __forceinline__ int ihist_bin_of_rank(const uint32_t *cum, int nb, uint32_t k) {
    int lo = 0, hi = nb - 1;  // smallest b with cum[b] > k
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cum[mid] > k) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__device__ SegStats seg_stats(ValCtx &C, int a, int b, int flags) {
    SegStats R;
    R.med = CUDART_NAN_F; R.mad = CUDART_NAN_F; R.lr = CUDART_NAN;
    clip_seg(a, b, C.src.n);
    const int n = b - a;
    if (n <= 0) return R;
    const bool fast = C.int_keys && (C.wkmax - C.wkmin) < (uint32_t)ADB_SEL_NB;
    if (!fast) {
        R.med = seg_median(C, a, b);
        if (flags & SS_MAD) R.mad = seg_mad(C, a, b, R.med);
        if (flags & SS_LR) R.lr = seg_local_range(C, a, b);
        return R;
    }
    const int T = blockDim.x, tid = threadIdx.x;
    uint32_t *hist = C.S.hist;
    const uint32_t kmin = C.wkmin;
    const int nb = (int)(C.wkmax - C.wkmin) + 1;
    const float coff = C.src.coff, cscale = C.src.cscale;
    const int16_t *p = C.src.i16 + a;
    __syncthreads();
    for (int q = tid; q < ADB_SEL_NB; q += T) hist[q] = 0;
    __syncthreads();
    {
        const uint32_t bias = 32768u - kmin;
        int j = tid;
        for (; j + 3 * T < n; j += 4 * T) {
            const int v0 = p[j], v1 = p[j + T], v2 = p[j + 2 * T], v3 = p[j + 3 * T];
            atomicAdd(&hist[(uint32_t)v0 + bias], 1u);
            atomicAdd(&hist[(uint32_t)v1 + bias], 1u);
            atomicAdd(&hist[(uint32_t)v2 + bias], 1u);
            atomicAdd(&hist[(uint32_t)v3 + bias], 1u);
        }
        for (; j < n; j += T) atomicAdd(&hist[(uint32_t)(int)p[j] + bias], 1u);
    }
    __syncthreads();
    // in-place inclusive scan over ADB_SEL_NB bins: contiguous chunk per thread + warp/block offsets
    {
        const int per = ADB_SEL_NB / T;  // 8 for 256 threads
        const int q0 = tid * per;
        uint32_t loc = 0;
        for (int q = q0; q < q0 + per; q++) { loc += hist[q]; hist[q] = loc; }
        uint32_t incl = loc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(ADB_FULL, incl, o);
            if ((tid & 31) >= o) incl += v;
        }
        if ((tid & 31) == 31) C.S.warp_tot[tid >> 5] = incl;
        __syncthreads();
        uint32_t wbase = 0;
        for (int w = 0; w < (tid >> 5); w++) wbase += C.S.warp_tot[w];
        const uint32_t add = wbase + incl - loc;
        if (add) for (int q = q0; q < q0 + per; q++) hist[q] += add;
    }
    __syncthreads();
    auto val = [&](int bin) { return __fmul_rn(__fadd_rn((float)((int)((uint32_t)bin + kmin) - 32768), coff), cscale); };
    // rank look-ups by six threads (median x2, percentile x4), results broadcast through shared memory
    float *fb = (float *)C.kbuf;  // 8 floats
    {
        const double v85 = __dmul_rn((double)(n - 1), 0.85), v15 = __dmul_rn((double)(n - 1), 0.15);
        const int l85 = (int)floor(v85), l15 = (int)floor(v15);
        if (tid < 6) {
            int rank;
            switch (tid) {
                case 0: rank = (n - 1) / 2; break;
                case 1: rank = n / 2; break;
                case 2: rank = l15; break;
                case 3: rank = min(l15 + 1, n - 1); break;
                case 4: rank = l85; break;
                default: rank = min(l85 + 1, n - 1); break;
            }
            if (tid < 2 || (flags & SS_LR)) fb[tid] = val(ihist_bin_of_rank(hist, nb, (uint32_t)rank));
        }
        __syncthreads();
        // median (SURVEY A.1): odd -> s[n/2]; even -> f32(f32(a+b)/2)
        R.med = (n & 1) ? fb[0] : __fdiv_rn(__fadd_rn(fb[0], fb[1]), 2.0f);
        if (flags & SS_LR)
            R.lr = __dsub_rn(np_lerp_f32(fb[4], fb[5], __dsub_rn(v85, (double)l85)),
                             np_lerp_f32(fb[2], fb[3], __dsub_rn(v15, (double)l15)));
    }
    if (flags & SS_MAD) {
        // k-th smallest deviation t* = min{ dev(code) : #(dev <= dev(code)) > k } over the occupied codes
        const float med = R.med;
        auto dev = [&](int bin) { return fabsf(__fsub_rn(val(bin), med)); };
        auto cum = [&](int x) -> uint32_t { return x < 0 ? 0u : hist[x]; };
        uint32_t *ub = C.kbuf + 6;  // 2 words: float bits of the answers (deviations are >= 0: bit order == value order)
        __syncthreads();
        if (tid == 0) { ub[0] = 0x7f800000u; ub[1] = 0x7f800000u; }
        int pv;  // first code whose value is >= med
        {
            int lo = 0, hi = nb;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (val(mid) >= med) hi = mid; else lo = mid + 1; }
            pv = lo;
        }
        __syncthreads();
        const uint32_t k0 = (uint32_t)((n - 1) / 2), k1 = (uint32_t)(n / 2);
        for (int bin = tid; bin < nb; bin += T) {
            if (cum(bin) == cum(bin - 1)) continue;  // empty code
            const float t = dev(bin);
            int lo = pv, hi = nb;  // right side [pv, nb): deviations non-decreasing -> first code with dev > t
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (dev(mid) > t) hi = mid; else lo = mid + 1; }
            const int r_gt = lo;
            lo = 0; hi = pv;       // left side [0, pv): deviations non-increasing -> first code with dev <= t
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (dev(mid) <= t) hi = mid; else lo = mid + 1; }
            const int l_le = lo;
            const uint32_t cnt_le = cum(r_gt - 1) - cum(l_le - 1);
            if (cnt_le > k0) atomicMin(&ub[0], __float_as_uint(t));
            if (cnt_le > k1) atomicMin(&ub[1], __float_as_uint(t));
        }
        __syncthreads();
        const float d0 = __uint_as_float(ub[0]), d1 = __uint_as_float(ub[1]);
        R.mad = (n & 1) ? d0 : __fdiv_rn(__fadd_rn(d0, d1), 2.0f);
    }
    __syncthreads();
    return R;
}

// float32 numpy mean of `n` samples starting at a, summed in numpy's pairwise order by one thread (the window is
// in shared memory).  Returns the mean to all threads.
__device__ float seg_mean_exact_small(ValCtx &C, int a, int n) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const ReadSrc &src = C.src;
        ((float *)C.dtmp)[0] = np_mean_f32([&](int i) { return src.pa(a + i); }, n);
    }
    __syncthreads();
    float r = ((float *)C.dtmp)[0];
    __syncthreads();
    return r;
}

// two means at once (real_range_check: first / last mean_window samples), threads 0 and 32
__device__ void seg_mean_exact_pair(ValCtx &C, int a0, int a1, int n, float &m0, float &m1) {
    __syncthreads();
    if (threadIdx.x == 0 || threadIdx.x == 32) {
        const ReadSrc &src = C.src;
        const int a = threadIdx.x == 0 ? a0 : a1;
        float s = np_sum_f32([&](int i) { return src.pa(a + i); }, n);
        ((float *)C.dtmp)[threadIdx.x == 0 ? 0 : 1] = __fdiv_rn(s, (float)n);
    }
    __syncthreads();
    m0 = ((float *)C.dtmp)[0];
    m1 = ((float *)C.dtmp)[1];
    __syncthreads();
}

// float32 np.var of n samples (numpy _var: mean, x - mean, x*x, pairwise sum / n)
__device__ float seg_var_exact_small(ValCtx &C, int a, int n) {
    float mean = seg_mean_exact_small(C, a, n);
    if (threadIdx.x == 0) {
        const ReadSrc &src = C.src;
        ((float *)C.dtmp)[0] = np_var_f32([&](int i) { return src.pa(a + i); }, n, mean);
    }
    __syncthreads();
    float r = ((float *)C.dtmp)[0];
    __syncthreads();
    return r;
}

// mean / population std of a segment for the partition table (signal_partitions.py:91-92).  numpy accumulates
// these in float32 pairwise order; they only have to agree to 1e-5 relative (north_star), so the sums are
// taken in float64 and rounded to float32 at the end.
__device__ void seg_mean_std(ValCtx &C, int a, int b, double &mean_out, double &std_out) {
    clip_seg(a, b, C.src.n);
    const int n = b - a;
    if (n <= 0) { mean_out = CUDART_NAN; std_out = CUDART_NAN; return; }
    const ReadSrc src = C.src;  // registers, not the context in local memory
    const int T = blockDim.x;
    if (src.i16) {
        // int16 sources: exact integer sums of the ADC codes (order-independent, hence the same bits whichever kernel
        // or launch geometry handles the read; identical to validate_fast_kernel).  numpy's float32 pairwise sums are
        // not reproduced -- the contract for mean / std is 1e-5 relative.
        const int16_t *p = src.i16 + a;
        long long s1 = 0, s2 = 0;
        for (int j = threadIdx.x; j < n; j += T) { const int c = p[j]; s1 += c; s2 += (long long)(c * c); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(ADB_FULL, s1, o); s2 += __shfl_xor_sync(ADB_FULL, s2, o); }
        long long *lt = reinterpret_cast<long long *>(C.dtmp);
        __syncthreads();
        if (threadIdx.x == 0) { lt[0] = 0; lt[1] = 0; }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) {
            atomicAdd((unsigned long long *)&lt[0], (unsigned long long)s1);
            atomicAdd((unsigned long long *)&lt[1], (unsigned long long)s2);
        }
        __syncthreads();
        const double mk = (double)lt[0] / n;
        double vk = (double)lt[1] / n - mk * mk;
        if (vk < 0) vk = 0;
        __syncthreads();
        mean_out = (double)(float)((mk + (double)src.coff) * (double)src.cscale);
        std_out = (double)(float)(sqrt(vk) * fabs((double)src.cscale));
        return;
    }
    double s = 0.0;
    if (src.i16) {
        const int16_t *p = src.i16 + a;
        const float co = src.coff, cs = src.cscale;
        for (int j = threadIdx.x; j < n; j += T) s += (double)__fmul_rn(__fadd_rn((float)p[j], co), cs);
    } else {
        const float *p = src.f32 + a;
        for (int j = threadIdx.x; j < n; j += T) s += (double)p[j];
    }
    s = warp_sum_d(s);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) C.dtmp[threadIdx.x >> 5] = s;
    __syncthreads();
    double tot = 0.0;
    for (int w = 0; w < (int)((blockDim.x + 31) >> 5); w++) tot += C.dtmp[w];
    const float mean32 = (float)(tot / n);
    __syncthreads();
    float qf = 0.f;  // per-thread partial in float32 (<= ~100 terms), combined in float64
    double q = 0.0;
    if (src.i16) {
        const int16_t *p = src.i16 + a;
        const float co = src.coff, cs = src.cscale;
        for (int j = threadIdx.x; j < n; j += T) { const float d = __fsub_rn(__fmul_rn(__fadd_rn((float)p[j], co), cs), mean32); qf = fmaf(d, d, qf); }
    } else {
        const float *p = src.f32 + a;
        for (int j = threadIdx.x; j < n; j += T) { const float d = __fsub_rn(p[j], mean32); qf = fmaf(d, d, qf); }
    }
    q = (double)qf;
    q = warp_sum_d(q);
    if ((threadIdx.x & 31) == 0) C.dtmp[threadIdx.x >> 5] = q;
    __syncthreads();
    double qt = 0.0;
    for (int w = 0; w < (int)((blockDim.x + 31) >> 5); w++) qt += C.dtmp[w];
    __syncthreads();
    mean_out = (double)mean32;
    std_out = (double)sqrtf((float)(qt / n));
}

// ---- bottleneck moving statistics (float32 recurrences, one lane each) --------------------------------------
// move_var(window wv) on thread 0 and move_mean(window wm) on thread 32 over src[a, a+L), reading the window from
// shared memory; the valid entries (index >= window-1) go, compacted, to series_a / series_b (global scratch).
// NaN-free segments (the only case real ADC data produces) take a branch-free loop whose only loop-carried
// dependencies are the float32 accumulators themselves; segments with NaN take the general path with bottleneck's
// count bookkeeping.  CTA-wide.
// NaN-free steps of the two recurrences, shared with the streaming session (adb_stream_session.cuh), which carries
// (amean, assqdm) and asum across pushes.  Warm-up of the variance: sample i < window enters Welford's update with a
// divide by i + 1; the first output clamps the running state and divides by the window.
__device__ __forceinline__ void mv_var_warm(float &amean, float &assqdm, float ai, int i) {
    const float delta = __fsub_rn(ai, amean);
    amean = __fadd_rn(amean, __fdiv_rn(delta, (float)(i + 1)));
    assqdm = __fadd_rn(assqdm, __fmul_rn(delta, __fsub_rn(ai, amean)));
}
__device__ __forceinline__ float mv_var_first(float &assqdm, int wv) {
    if (assqdm < 0) assqdm = 0;
    return __fdiv_rn(assqdm, (float)wv);
}
// sample ai enters, aold (window samples back) leaves; the output is assqdm * count_inv
__device__ __forceinline__ void mv_var_step(float &amean, float &assqdm, float ai, float aold, float count_inv) {
    const float delta = __fsub_rn(ai, aold);
    aold = __fsub_rn(aold, amean);
    amean = __fadd_rn(amean, __fmul_rn(delta, count_inv));
    ai = __fsub_rn(ai, amean);
    assqdm = __fadd_rn(assqdm, __fmul_rn(__fadd_rn(ai, aold), delta));
    if (assqdm < 0) assqdm = 0;
}
// running sum of the moving mean past its first window; the output is asum * count_inv
__device__ __forceinline__ float mv_mean_step(float asum, float ai, float aold) { return __fadd_rn(asum, __fsub_rn(ai, aold)); }

__device__ void seg_moving_stats(ValCtx &C, int a, int L, int wv, int wm, bool do_var, bool do_mean) {
    const ReadSrc &src = C.src;
    // any NaN in the segment?
    __syncthreads();
    if (threadIdx.x == 0) C.itmp[6] = 0;
    __syncthreads();
    {
        bool bad = false;
        for (int j = threadIdx.x; j < L; j += blockDim.x) { float v = src.pa(a + j); bad |= !(v == v); }
        if (bad) C.itmp[6] = 1;
    }
    __syncthreads();
    const bool has_nan = C.itmp[6] != 0;
    if (threadIdx.x == 0 && do_var) {
        float *y = C.series_a;
        if (!has_nan) {
            float amean = 0.f, assqdm = 0.f;
            for (int i = 0; i < wv; i++) mv_var_warm(amean, assqdm, src.pa(a + i), i);
            y[0] = mv_var_first(assqdm, wv);
            const float count_inv = (float)(1.0 / (double)wv);
#pragma unroll 4
            for (int i = wv; i < L; i++) {
                mv_var_step(amean, assqdm, src.pa(a + i), src.pa(a + i - wv), count_inv);
                y[i - (wv - 1)] = __fmul_rn(assqdm, count_inv);
            }
        } else {
            int count = 0;
            float amean = 0.f, assqdm = 0.f, count_inv = 0.f, ddof_inv = 0.f;
            for (int i = 0; i < L; i++) {
                float ai = src.pa(a + i), yi;
                if (i < wv) {
                    if (ai == ai) {
                        count += 1;
                        const float delta = __fsub_rn(ai, amean);
                        amean = __fadd_rn(amean, __fdiv_rn(delta, (float)count));
                        assqdm = __fadd_rn(assqdm, __fmul_rn(delta, __fsub_rn(ai, amean)));
                    }
                    if (i == wv - 1) {
                        if (count >= wv) { if (assqdm < 0) assqdm = 0; yi = __fdiv_rn(assqdm, (float)count); }
                        else yi = CUDART_NAN_F;
                        y[0] = yi;
                        count_inv = (float)(1.0 / (double)count);
                        ddof_inv = count_inv;
                    }
                } else {
                    float aold = src.pa(a + i - wv);
                    if (ai == ai) {
                        if (aold == aold) {
                            const float delta = __fsub_rn(ai, aold);
                            aold = __fsub_rn(aold, amean);
                            amean = __fadd_rn(amean, __fmul_rn(delta, count_inv));
                            ai = __fsub_rn(ai, amean);
                            assqdm = __fadd_rn(assqdm, __fmul_rn(__fadd_rn(ai, aold), delta));
                        } else {
                            count++;
                            count_inv = (float)(1.0 / (double)count);
                            ddof_inv = count_inv;
                            const float delta = __fsub_rn(ai, amean);
                            amean = __fadd_rn(amean, __fmul_rn(delta, count_inv));
                            assqdm = __fadd_rn(assqdm, __fmul_rn(delta, __fsub_rn(ai, amean)));
                        }
                    } else if (aold == aold) {
                        count--;
                        count_inv = (float)(1.0 / (double)count);
                        ddof_inv = count_inv;
                        if (count > 0) {
                            const float delta = __fsub_rn(aold, amean);
                            amean = __fsub_rn(amean, __fmul_rn(delta, count_inv));
                            assqdm = __fsub_rn(assqdm, __fmul_rn(delta, __fsub_rn(aold, amean)));
                        } else { amean = 0; assqdm = 0; }
                    }
                    if (count >= wv) { if (assqdm < 0) assqdm = 0; yi = __fmul_rn(assqdm, ddof_inv); }
                    else yi = CUDART_NAN_F;
                    y[i - (wv - 1)] = yi;
                }
            }
        }
    }
    if (threadIdx.x == 32 && do_mean) {
        float *y = C.series_b;
        if (!has_nan) {
            float asum = 0.f;
            for (int i = 0; i < wm; i++) asum = __fadd_rn(asum, src.pa(a + i));
            y[0] = __fdiv_rn(asum, (float)wm);
            const float count_inv = (float)(1.0 / (double)wm);
#pragma unroll 8
            for (int i = wm; i < L; i++) {
                asum = mv_mean_step(asum, src.pa(a + i), src.pa(a + i - wm));
                y[i - (wm - 1)] = __fmul_rn(asum, count_inv);
            }
        } else {
            int count = 0;
            float asum = 0.f, count_inv = 0.f;
            for (int i = 0; i < L; i++) {
                const float ai = src.pa(a + i);
                if (i < wm) {
                    if (ai == ai) { asum = __fadd_rn(asum, ai); count += 1; }
                    if (i == wm - 1) {
                        y[0] = (count >= wm) ? __fdiv_rn(asum, (float)count) : CUDART_NAN_F;
                        count_inv = (float)(1.0 / (double)count);
                    }
                } else {
                    const float aold = src.pa(a + i - wm);
                    if (ai == ai) {
                        if (aold == aold) asum = __fadd_rn(asum, __fsub_rn(ai, aold));
                        else { asum = __fadd_rn(asum, ai); count++; count_inv = (float)(1.0 / (double)count); }
                    } else if (aold == aold) {
                        asum = __fsub_rn(asum, aold); count--; count_inv = (float)(1.0 / (double)count);
                    }
                    y[i - (wm - 1)] = (count >= wm) ? __fmul_rn(asum, count_inv) : CUDART_NAN_F;
                }
            }
        }
    }
    __threadfence_block();
    __syncthreads();
}

// ---- thread-per-read moving statistics -------------------------------------------------------------------------
// The two bottleneck recurrences are strictly sequential in float32 (each output depends on every earlier sample),
// but reads are independent: one THREAD per read runs both recurrences over [ae, pe) straight from global memory
// (the lagging a[i-window] stream hits L1/L2) and writes the valid entries of both series to a per-read scratch row.
// Only NaN-free segments are handled here (real ADC data); anything else, and candidates other than the first,
// falls back to the in-CTA path above.  Conditions mirror mvs.py:76-107.
struct MvsSeriesArgs {
    BatchDev B;
    const int *given;
    int given_stride;
    int n_reads;
    float *var_pool;          // [pool_cap] compact rows of moving variance
    float *mean_pool;         // [pool_cap] compact rows of moving mean (same offsets)
    long long pool_cap;       // floats per pool
    unsigned long long *cursor;  // allocation cursor (zeroed before the launch)
    long long *row_off;       // [n_reads] offset of the read's row in the pools, or -1 (not precomputed)
    int *meta;                // [n_reads][2] = ae, pe the row belongs to
    const int *perm;          // optional [n_reads]: lane q works on read perm[q] (reads sorted by segment length)
    // second pass (reads the counting-based validate kernel handed over): only the first *n_active entries of perm are
    // reads, and the series run up to the LARGEST poly(A) candidate -- the recurrences start at adapter_end, so the
    // series of every smaller candidate (and of the hail-mary poly(A) end) is a prefix of that row
    const int *n_active;      // optional device counter
    int all_cands;            // 1: polya_end = max over the read's non-zero candidates
    int n_cand;               // candidates per read in `given` (after adapter_end) when ntopk_per_read == nullptr
    const int *ntopk_per_read;
};

// reads still to be validated after validate_fast_kernel -> compact list (order irrelevant: rows are independent)
__global__ void mvs_pending_kernel(const unsigned char *done, int n_reads, int *list, int *count) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool p = r < n_reads && done[r] != 1;  // (2 = first candidate settled by the fast kernel, the others pending)
    const unsigned m = __ballot_sync(ADB_FULL, p);
    if (!m) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(ADB_FULL, base, 0);
    if (p) list[base + __popc(m & ((1u << lane) - 1))] = r;
}

struct __align__(16) MvsRow {  // per-read constants of the transposing phases, read as shared-memory broadcasts
    const int16_t *rp;        // first sample of the segment
    float *gvp, *gmp;         // output rows, pre-shifted: entry i of the series lives at gvp[i] / gmp[i]
    int L, iminv, iminm, pad; // segment length; first valid index of either series (INT_MAX: series not wanted)
};
#define MVS_LANES 128   // reads per CTA (one lane each; every warp works on its own 32 reads, no CTA-wide sync)
#define MVS_C 32        // samples staged per step
#define MVS_RING 256    // circular input columns per read (>= window + 2 * MVS_C), power of two
#define MVS_RING_STRIDE 257  // float units, odd -> lanes walking their own row hit distinct banks
#define MVS_OUT_STRIDE 33    // float units
#define MVS_MAX_WINDOW (MVS_RING - 2 * MVS_C)

__host__ __device__ inline size_t mvs_smem_bytes() {
    return (size_t)MVS_LANES * MVS_RING_STRIDE * 4 + 2 * (size_t)MVS_LANES * MVS_OUT_STRIDE * 4 + (size_t)MVS_LANES * 8 +
           (size_t)MVS_LANES * sizeof(MvsRow) + 64;
}

// eligibility of a read for the precomputed series (mirrors the early exits of mvs.py:76-107)
__device__ __forceinline__ bool mvs_plan(const adb_config &cfg, const ReadSrc &src, int ae, int pe, int &a, int &L,
                                         bool &win_var, bool &win_mean) {
    if (!cfg.mvs_detect_check) return false;
    const int size = src.n;
    if (pe == 0 || ae == 0 || pe < ae || pe - ae <= 2) return false;
    if (size < ae + cfg.median_shift_window) return false;
    win_var = !(pe - ae <= cfg.pA_var_window + 2);
    win_mean = !(pe - ae <= cfg.pA_mean_window + 2);
    if (!win_var && !win_mean) return false;
    a = min(ae, size);
    L = min(pe, size) - a;
    if (L < max(cfg.pA_var_window, cfg.pA_mean_window)) return false;
    return true;
}

// int16 sources: one lane per read, 32 reads per warp, warps independent of each other.  Per step of MVS_C samples a
// warp (1) issues the coalesced row loads of the NEXT step into registers, (2) lets every lane advance its two
// recurrences over the current step from its own row of a shared-memory ring of CALIBRATED samples (circular history
// for a[i - window]), (3) writes the step's outputs row by row (coalesced) from a shared tile, (4) calibrates and
// parks the prefetched samples in the ring.  A read's time is its segment length times the cycles per sample of (2)
// -- the kernel's duration is that of its longest read -- so the steady state of (2) is branch-free and unrolled:
// the loads and the differences a[i] - a[i - window] of eight samples are independent of the recurrences, what stays
// loop-carried is one addition per sample for each running mean and an add + clamp for the sum of squares.
__global__ void __launch_bounds__(MVS_LANES) mvs_series_kernel(MvsSeriesArgs A, adb_config cfg) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *ring = (float *)smem + (size_t)warp * 32 * MVS_RING_STRIDE;
    float *ov = (float *)smem + (size_t)MVS_LANES * MVS_RING_STRIDE + warp * 32 * MVS_OUT_STRIDE;
    float *om = ov + MVS_LANES * MVS_OUT_STRIDE;
    float2 *cal_all = (float2 *)((float *)smem + (size_t)MVS_LANES * MVS_RING_STRIDE + 2 * MVS_LANES * MVS_OUT_STRIDE);
    float2 *cal = cal_all + warp * 32;
    MvsRow *tab = (MvsRow *)(cal_all + MVS_LANES) + warp * 32;
    const int qi = blockIdx.x * MVS_LANES + tid;
    const int n_lim = A.n_active ? min(*A.n_active, A.n_reads) : A.n_reads;
    const int q = (qi < n_lim) ? (A.perm ? A.perm[qi] : qi) : A.n_reads;
    const int wv = cfg.pA_var_window, wm = cfg.pA_mean_window;
    bool active = false, win_var = false, win_mean = false;
    int a = 0, L = 0, ae = 0, pe = 0;
    float coff = 0.f, cscale = 1.f;
    const int16_t *rp = nullptr;
    if (q < A.n_reads) {
        const int *g = A.given + (size_t)q * A.given_stride;
        ae = g[0]; pe = g[1];
        if (A.all_cands) {  // the candidates the reference's loop can reach (combined.py:464-466: stops at the first 0)
            const int nt = A.ntopk_per_read ? A.ntopk_per_read[q] : A.n_cand;
            for (int t = 0; t < nt && g[1 + t] != 0; t++) pe = max(pe, g[1 + t]);
        }
        const ReadSrc src = make_src(A.B, q);
        active = (src.i16 != nullptr) && wv <= MVS_MAX_WINDOW && wm <= MVS_MAX_WINDOW &&
                 mvs_plan(cfg, src, ae, pe, a, L, win_var, win_mean) && isfinite(src.coff) && isfinite(src.cscale);
        coff = src.coff; cscale = src.cscale;
        if (active) rp = src.i16 + a;
    }
    // compact row allocation: warp-level exclusive scan of the (4-float aligned) row lengths + one atomic per warp
    const int need = active ? ((L + 3) & ~3) : 0;
    int incl = need;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(ADB_FULL, incl, o);
        if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(ADB_FULL, incl, 31);
    long long base = 0;
    if (lane == 0 && total > 0) base = (long long)atomicAdd(A.cursor, (unsigned long long)total);
    base = __shfl_sync(ADB_FULL, base, 0);
    const long long myoff = base + incl - need;
    if (active && myoff + need > A.pool_cap) active = false;  // pool exhausted: the validate kernel falls back
    if (q < A.n_reads) {
        A.row_off[q] = active ? myoff : -1;
        A.meta[2 * (size_t)q] = active ? ae : -1;
        A.meta[2 * (size_t)q + 1] = active ? pe : -1;
    }
    if (!active) { L = 0; rp = nullptr; }
    int Lmax = L;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) Lmax = max(Lmax, __shfl_xor_sync(ADB_FULL, Lmax, o));
    if (Lmax == 0) return;
    cal[lane] = make_float2(coff, cscale);
    const int flag = (win_var ? 1 : 0) | (win_mean ? 2 : 0);
    float amean = 0.f, assqdm = 0.f, asum = 0.f;
    const float cinv_v = (float)(1.0 / (double)wv), cinv_m = (float)(1.0 / (double)wm);
    const float *myrow = ring + (size_t)lane * MVS_RING_STRIDE;
    float *myov = ov + lane * MVS_OUT_STRIDE, *myom = om + lane * MVS_OUT_STRIDE;
    const int wmax = max(wv, wm);
    {
        MvsRow t;
        t.rp = rp;
        t.gvp = A.var_pool + myoff - (wv - 1);
        t.gmp = A.mean_pool + myoff - (wm - 1);
        t.L = L;
        t.iminv = (flag & 1) ? wv - 1 : 0x7fffffff;
        t.iminm = (flag & 2) ? wm - 1 : 0x7fffffff;
        t.pad = 0;
        tab[lane] = t;
    }
    // steps inside [wmax, Lmin) need no per-row tests when every row wants both series
    int Lmin = L;
    bool both = flag == 3;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) Lmin = min(Lmin, __shfl_xor_sync(ADB_FULL, Lmin, o));
    both = __all_sync(ADB_FULL, both);
    if (!both) Lmin = 0;
    // prefetch registers: sample (base + lane) of every row
    int16_t pf[32];
    auto prefetch = [&](int step_base) {
        const int i = step_base + lane;
        if (step_base + MVS_C <= Lmin) {
#pragma unroll
            for (int row = 0; row < 32; row++) pf[row] = __ldg(tab[row].rp + i);
        } else {
#pragma unroll
            for (int row = 0; row < 32; row++) {
                const int16_t *p = tab[row].rp;
                pf[row] = (i < tab[row].L) ? __ldg(p + i) : (int16_t)0;
            }
        }
    };
    auto park = [&](int step_base) {  // pA = (adc + offset) * scale, each step rounded to float32
        const int col = (step_base + lane) & (MVS_RING - 1);
#pragma unroll
        for (int row = 0; row < 32; row++) {
            const float2 c = cal[row];
            ring[(size_t)row * MVS_RING_STRIDE + col] = __fmul_rn(__fadd_rn((float)pf[row], c.x), c.y);
        }
    };
    __syncwarp();
    prefetch(0);
    park(0);
    __syncwarp();
    for (int base_i = 0; base_i < Lmax; base_i += MVS_C) {
        const bool more = base_i + MVS_C < Lmax;
        if (more) prefetch(base_i + MVS_C);  // loads in flight while the recurrences run
        if (base_i >= wmax) {
            // steady state (every window is full); lanes past their own end compute on zeros, nothing of it is stored
#pragma unroll
            for (int g = 0; g < MVS_C; g += 8) {
                float x[8], xv[8], xm[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = base_i + g + u;
                    x[u] = myrow[i & (MVS_RING - 1)];
                    xv[u] = myrow[(i - wv) & (MVS_RING - 1)];
                    xm[u] = myrow[(i - wm) & (MVS_RING - 1)];
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    asum = __fadd_rn(asum, __fsub_rn(x[u], xm[u]));
                    myom[g + u] = __fmul_rn(asum, cinv_m);
                    const float delta = __fsub_rn(x[u], xv[u]);
                    const float ao = __fsub_rn(xv[u], amean);
                    amean = __fadd_rn(amean, __fmul_rn(delta, cinv_v));
                    const float ai = __fsub_rn(x[u], amean);
                    assqdm = __fadd_rn(assqdm, __fmul_rn(__fadd_rn(ai, ao), delta));
                    assqdm = (assqdm < 0.f) ? 0.f : assqdm;
                    myov[g + u] = __fmul_rn(assqdm, cinv_v);
                }
            }
        } else if (base_i < L) {
            const int iend = min(base_i + MVS_C, L);
            for (int i = base_i; i < iend; i++) {
                const float x = myrow[i & (MVS_RING - 1)];
                if (win_var) {
                    if (i < wv) {
                        const float delta = __fsub_rn(x, amean);
                        amean = __fadd_rn(amean, __fdiv_rn(delta, (float)(i + 1)));
                        assqdm = __fadd_rn(assqdm, __fmul_rn(delta, __fsub_rn(x, amean)));
                        if (i == wv - 1) {
                            if (assqdm < 0) assqdm = 0;
                            myov[i - base_i] = __fdiv_rn(assqdm, (float)wv);
                        }
                    } else {
                        float ai = x;
                        float aold = myrow[(i - wv) & (MVS_RING - 1)];
                        const float delta = __fsub_rn(ai, aold);
                        aold = __fsub_rn(aold, amean);
                        amean = __fadd_rn(amean, __fmul_rn(delta, cinv_v));
                        ai = __fsub_rn(ai, amean);
                        assqdm = __fadd_rn(assqdm, __fmul_rn(__fadd_rn(ai, aold), delta));
                        if (assqdm < 0) assqdm = 0;
                        myov[i - base_i] = __fmul_rn(assqdm, cinv_v);
                    }
                }
                if (win_mean) {
                    if (i < wm) {
                        asum = __fadd_rn(asum, x);
                        if (i == wm - 1) myom[i - base_i] = __fdiv_rn(asum, (float)wm);
                    } else {
                        const float aold = myrow[(i - wm) & (MVS_RING - 1)];
                        asum = __fadd_rn(asum, __fsub_rn(x, aold));
                        myom[i - base_i] = __fmul_rn(asum, cinv_m);
                    }
                }
            }
        }
        __syncwarp();
        // ---- coalesced row stores of the valid entries ----
        {
            const int i = base_i + lane;
            if (base_i >= wmax && base_i + MVS_C <= Lmin) {
#pragma unroll 8
                for (int row = 0; row < 32; row++) {
                    const MvsRow t = tab[row];
                    t.gvp[i] = ov[row * MVS_OUT_STRIDE + lane];
                    t.gmp[i] = om[row * MVS_OUT_STRIDE + lane];
                }
            } else {
#pragma unroll 4
                for (int row = 0; row < 32; row++) {
                    const MvsRow t = tab[row];
                    if (i < t.L) {
                        if (i >= t.iminv) t.gvp[i] = ov[row * MVS_OUT_STRIDE + lane];
                        if (i >= t.iminm) t.gmp[i] = om[row * MVS_OUT_STRIDE + lane];
                    }
                }
            }
        }
        if (more) park(base_i + MVS_C);
        __syncwarp();
    }
}

// ---- reads sorted by the length of their moving-statistics segment -------------------------------------------------
// A warp of mvs_series_kernel runs as long as its longest read, so reads of similar length are put into the same
// warp: counting sort by length bucket (64 samples), longest first; reads without a segment come last.
#define MVS_NBUCKET 512
__device__ __forceinline__ int mvs_len_bucket(const MvsSeriesArgs &A, const adb_config &cfg, int r) {
    const int *g = A.given + (size_t)r * A.given_stride;
    const ReadSrc src = make_src(A.B, r);
    int a, L;
    bool wv_, wm_;
    if (src.i16 == nullptr || !mvs_plan(cfg, src, g[0], g[1], a, L, wv_, wm_)) return MVS_NBUCKET - 1;
    return max(MVS_NBUCKET - 2 - min(L >> 6, MVS_NBUCKET - 2), 0);  // longest first
}
__global__ void mvs_len_hist_kernel(MvsSeriesArgs A, adb_config cfg, int *bucket_cnt) {
    __shared__ int sh[MVS_NBUCKET];
    for (int b = threadIdx.x; b < MVS_NBUCKET; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < A.n_reads; r += gridDim.x * blockDim.x)
        atomicAdd(&sh[mvs_len_bucket(A, cfg, r)], 1);
    __syncthreads();
    for (int b = threadIdx.x; b < MVS_NBUCKET; b += blockDim.x) if (sh[b]) atomicAdd(&bucket_cnt[b], sh[b]);
}
__global__ void mvs_len_scan_kernel(int *bucket_cnt /* in: counts, out: running cursors = start offsets */) {
    __shared__ int sh[MVS_NBUCKET];
    const int t = threadIdx.x;  // MVS_NBUCKET threads
    sh[t] = bucket_cnt[t];
    __syncthreads();
    for (int o = 1; o < MVS_NBUCKET; o <<= 1) {
        const int v = (t >= o) ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += v;
        __syncthreads();
    }
    bucket_cnt[t] = sh[t] - bucket_cnt[t];  // exclusive prefix
}
__global__ void mvs_len_scatter_kernel(MvsSeriesArgs A, adb_config cfg, int *bucket_cursor, int *perm) {
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < A.n_reads; r += gridDim.x * blockDim.x)
        perm[atomicAdd(&bucket_cursor[mvs_len_bucket(A, cfg, r)], 1)] = r;
}

// float32 sources (the reference seam): one thread per read straight from global memory.  This path is PCIe-bound
// anyway (106 MB per minibatch over the bus), so it keeps the simple form.
__global__ void __launch_bounds__(128) mvs_series_f32_kernel(MvsSeriesArgs A, adb_config cfg) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= A.n_reads) return;
    const int r = q;
    int *meta = A.meta + 2 * (size_t)q;
    meta[0] = -1;
    meta[1] = -1;
    A.row_off[q] = -1;
    const int *g = A.given + (size_t)r * A.given_stride;
    const int ae = g[0], pe = g[1];
    const ReadSrc src = make_src(A.B, r);
    if (!src.f32) return;
    int a, L;
    bool win_var, win_mean;
    if (!mvs_plan(cfg, src, ae, pe, a, L, win_var, win_mean)) return;
    const int wv = cfg.pA_var_window, wm = cfg.pA_mean_window;
    const float *__restrict__ x = src.f32 + a;
    for (int i = 0; i < L; i++) { float v = x[i]; if (!(v == v)) return; }
    const int need = (L + 3) & ~3;
    const long long off = (long long)atomicAdd(A.cursor, (unsigned long long)need);
    if (off + need > A.pool_cap) return;
    A.row_off[q] = off;
    float *__restrict__ yv = A.var_pool + off;
    float *__restrict__ ym = A.mean_pool + off;
    const float cinv_v = (float)(1.0 / (double)wv), cinv_m = (float)(1.0 / (double)wm);
    if (win_var) {
        float amean = 0.f, assqdm = 0.f;
        for (int i = 0; i < wv; i++) {
            const float ai = x[i];
            const float delta = __fsub_rn(ai, amean);
            amean = __fadd_rn(amean, __fdiv_rn(delta, (float)(i + 1)));
            assqdm = __fadd_rn(assqdm, __fmul_rn(delta, __fsub_rn(ai, amean)));
        }
        if (assqdm < 0) assqdm = 0;
        yv[0] = __fdiv_rn(assqdm, (float)wv);
#pragma unroll 4
        for (int i = wv; i < L; i++) {
            float ai = x[i], aold = x[i - wv];
            const float delta = __fsub_rn(ai, aold);
            aold = __fsub_rn(aold, amean);
            amean = __fadd_rn(amean, __fmul_rn(delta, cinv_v));
            ai = __fsub_rn(ai, amean);
            assqdm = __fadd_rn(assqdm, __fmul_rn(__fadd_rn(ai, aold), delta));
            if (assqdm < 0) assqdm = 0;
            yv[i - (wv - 1)] = __fmul_rn(assqdm, cinv_v);
        }
    }
    if (win_mean) {
        float asum = 0.f;
        for (int i = 0; i < wm; i++) asum = __fadd_rn(asum, x[i]);
        ym[0] = __fdiv_rn(asum, (float)wm);
#pragma unroll 4
        for (int i = wm; i < L; i++) {
            asum = __fadd_rn(asum, __fsub_rn(x[i], x[i - wm]));
            ym[i - (wm - 1)] = __fmul_rn(asum, cinv_m);
        }
    }
    meta[0] = ae;
    meta[1] = pe;
}

// keys of a float32 series that may contain NaN: NaNs sort last (key 0xffffffff) and are not counted
struct BufKeysNan {
    const float *p;
    __device__ __forceinline__ uint32_t operator()(int j) const { float v = p[j]; return (v == v) ? f32_key(v) : 0xffffffffu; }
};

// np.nanmedian of a float32 series in global scratch: NaNs are dropped (they get the largest key and the ranks
// are taken among the non-NaN count)
__device__ float series_nanmedian(ValCtx &C, const float *p, int n) {
    if (n <= 0) return CUDART_NAN_F;
    __syncthreads();
    if (threadIdx.x == 0) C.itmp[7] = 0;
    __syncthreads();
    int cnt = 0;
    // int16 sources with a finite calibration have no NaN samples, so neither have their moving statistics
    const bool nan_free = C.src.i16 != nullptr && isfinite(C.src.coff) && isfinite(C.src.cscale);
    if (nan_free) {
        if (threadIdx.x == 0) C.itmp[7] = n;
    } else {
        const int T = blockDim.x;
        int j = threadIdx.x;
        for (; j + 3 * T < n; j += 4 * T) {
            const float v0 = p[j], v1 = p[j + T], v2 = p[j + 2 * T], v3 = p[j + 3 * T];
            cnt += (v0 == v0) + (v1 == v1) + (v2 == v2) + (v3 == v3);
        }
        for (; j < n; j += T) { const float v = p[j]; cnt += (v == v); }
    }
    cnt = warp_sum_i(cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&C.itmp[7], cnt);
    __syncthreads();
    const int nvalid = C.itmp[7];
    __syncthreads();
    if (nvalid == 0) return CUDART_NAN_F;
    BufKeysNan K{p};
    uint32_t kmin, kmax;
    cta_key_minmax(K, n, kmin, kmax, C.S);
    int *ranks = (int *)(C.kbuf + 4);
    if (threadIdx.x == 0) { ranks[0] = (nvalid - 1) / 2; ranks[1] = nvalid / 2; }
    __syncthreads();
    cta_select_ranks(K, n, kmin, kmax, ranks, (nvalid & 1) ? 1 : 2, C.kbuf, C.S);
    const float x0 = key_f32(C.kbuf[0]);
    if (nvalid & 1) return x0;
    return __fdiv_rn(__fadd_rn(x0, key_f32(C.kbuf[1])), 2.0f);
}

// ---- mean_var_shift_polyA_check (mvs.py:45-158) -------------------------------------------------------------
struct MvsOut {
    bool ok;
    int fail_mask;   // bit i: check i failed (mean var med range shift)
    double v[5];     // mean, var, med, local_range, med_shift (all 0 on early fail)
    float polya_mad; // MAD of signal[ae:pe) from the same histogram (reused by the partition table)
};

__device__ MvsOut mvs_check(ValCtx &C, int ae, int pe, double mean_lo, double mean_hi) {
    const adb_config &cfg = *C.cfg;
    MvsOut R;
    R.ok = false; R.fail_mask = 0x1f; R.polya_mad = 0.f;
    for (int i = 0; i < 5; i++) R.v[i] = 0.0;
    const int size = C.src.n;
    if (pe == 0 || ae == 0 || pe < ae || pe - ae <= 2) return R;
    if (size < ae + cfg.median_shift_window) return R;
    int a = ae, b = pe;
    clip_seg(a, b, size);
    const int L = b - a;
    float var32, mean32;
    const bool win_var = !(pe - ae <= cfg.pA_var_window + 2);
    const bool win_mean = !(pe - ae <= cfg.pA_mean_window + 2);
    // a precomputed row serves every poly(A) end up to its own: the series of [ae, pe) is a prefix of the row
    const bool pre = (C.pre_var != nullptr) && C.pre_ae == ae && pe <= C.pre_pe;
    if (!pre && (win_var || win_mean))
        seg_moving_stats(C, a, L, cfg.pA_var_window, cfg.pA_mean_window, win_var, win_mean);
    if (win_var) var32 = series_nanmedian(C, pre ? C.pre_var : C.series_a, L - (cfg.pA_var_window - 1));
    else var32 = seg_var_exact_small(C, a, L);
    if (win_mean) mean32 = series_nanmedian(C, pre ? C.pre_mean : C.series_b, L - (cfg.pA_mean_window - 1));
    else mean32 = seg_mean_exact_small(C, a, L);
    const SegStats P = seg_stats(C, ae, pe, SS_MED | SS_LR | SS_MAD);
    const float med32 = P.med;
    const double lr = P.lr;
    R.polya_mad = P.mad;
    const float m_after = seg_stats(C, ae, min(ae + cfg.median_shift_window, size), SS_MED).med;
    const float m_before = seg_stats(C, max(ae - cfg.median_shift_window, 0), ae, SS_MED).med;
    const float shift32 = __fsub_rn(m_after, m_before);
    R.v[0] = (double)mean32; R.v[1] = (double)var32; R.v[2] = (double)med32; R.v[3] = lr; R.v[4] = (double)shift32;
    const double mr[2] = {mean_lo, mean_hi};
    R.fail_mask = vc_mvs_mask(cfg, R.v, mr);
    R.ok = (R.fail_mask == 0);
    return R;
}

// ---- mean_var_shift_polyA_detect_at_loc (mvs.py:181-338, less_signal_ok=False) -------------------------------
// The poly(A) start is looked for in [loc, loc + search_window): bottleneck move_mean / move_var over
// signal[loc - offset : loc + search_window) (offset = the larger window), first position where both are in range.
struct MvsLocOut {
    bool ok;
    int idx;      // mvs_adapter_end (0: nothing found)
    double v[5];  // mean, var at the found position (or at loc + offset), polya med, local range, med shift
};

__device__ MvsLocOut mvs_detect_at_loc(ValCtx &C, int loc, double mean_lo, double mean_hi, bool mean_bounds_f64) {
    const adb_config &cfg = *C.cfg;
    MvsLocOut R;
    R.ok = false; R.idx = 0;
    for (int i = 0; i < 5; i++) R.v[i] = 0.0;
    const int size = C.src.n;
    const int wm = cfg.pA_mean_window, wv = cfg.pA_var_window, sw = cfg.search_window;
    if (size < loc + sw + max(cfg.median_shift_window, cfg.polyA_window)) return R;  // mvs.py:238-254
    const int offset = max(wm, wv);
    if (loc < offset) return R;                                                     // mvs.py:257-269
    const int a = loc - offset, L = offset + sw;
    seg_moving_stats(C, a, L, wv, wm, true, true);
    // series_a[j] = move_var[j + wv - 1], series_b[j] = move_mean[j + wm - 1]; the first offset-1 entries of at
    // least one series are NaN (never in range).  in_range on a float32 array (utils.py:16-28) compares in float32
    // against python-float bounds (numpy casts the weak scalar) and in float64 against np.float64 bounds, which is
    // what pA_mean_range holds once it is derived from the adapter median (combined.py:447-458).
    const float vlo = (float)cfg.pA_var_range[0], vhi = (float)cfg.pA_var_range[1];
    const float mlo32 = (float)mean_lo, mhi32 = (float)mean_hi;
    __syncthreads();
    if (threadIdx.x == 0) C.itmp[7] = 0x7fffffff;
    __syncthreads();
    for (int i = offset - 1 + (int)threadIdx.x; i < L; i += blockDim.x) {
        const float mm = C.series_b[i - (wm - 1)], mv = C.series_a[i - (wv - 1)];
        const bool mean_ok = mean_bounds_f64 ? (mean_lo <= (double)mm && (double)mm <= mean_hi) : (mlo32 <= mm && mm <= mhi32);
        if (mean_ok && vlo <= mv && mv <= vhi) { atomicMin(&C.itmp[7], i); break; }
    }
    __syncthreads();
    int idx = C.itmp[7];
    if (idx == 0x7fffffff) idx = 0;  // np.argmax of an all-False mask
    float mean32, var32;
    if (idx > 0) {
        mean32 = C.series_b[idx - (wm - 1)]; var32 = C.series_a[idx - (wv - 1)];
        idx += loc - offset;
    } else {  // mvs.py:288-291: the features at loc (running-window lag = offset)
        mean32 = C.series_b[2 * offset - (wm - 1)]; var32 = C.series_a[2 * offset - (wv - 1)];
    }
    __syncthreads();
    const int loc_ = max(loc, idx);
    const SegStats P = seg_stats(C, loc_, min(loc_ + cfg.polyA_window, size), SS_MED | SS_LR);
    const float m_after = seg_stats(C, loc_, min(loc_ + cfg.median_shift_window, size), SS_MED).med;
    const float m_before = seg_stats(C, 0, loc_, SS_MED).med;
    R.idx = idx;
    R.v[0] = (double)mean32; R.v[1] = (double)var32; R.v[2] = (double)P.med; R.v[3] = P.lr;
    R.v[4] = (double)__fsub_rn(m_after, m_before);
    R.ok = idx > 0 && in_range_d(R.v[2], cfg.polyA_med_range) && in_range_d(R.v[3], cfg.polyA_local_range) &&
           in_range_d(R.v[4], cfg.median_shift_range);
    return R;
}

// ---- find_open_pores (anomalies.py:15-35) on signal[a:b), absolute indices ------------------------------------
// Returns the number of reported positions; *last = open_pores[-1]; the first ADB_MAX_OPEN_PORES go to rec.
__device__ int open_pores_scan(ValCtx &C, int a, int b, adb_record *rec, int *last) {
    clip_seg(a, b, C.src.n);
    const int n = b - a;
    const int T = blockDim.x, tid = threadIdx.x;
    const int chunk = (n + T - 1) / T;
    const int j0 = min(tid * chunk, n), j1 = min(j0 + chunk, n);
    int *sh = C.itmp;  // [0]=hits [1]=first hit [2]=last hit [3]=valid count [4]=last valid
    __syncthreads();
    if (tid == 0) { sh[0] = 0; sh[1] = 0x7fffffff; sh[2] = -1; sh[3] = 0; sh[4] = -1; }
    __syncthreads();
    // pass 1: hits, and "gap >= 10 to the previous hit" candidates (first-hit exclusion applied later)
    int hits = 0, first = 0x7fffffff, lastp = -1, ncand = 0, lastc = -1;
    for (int j = j0; j < j1; j++) {
        float v = C.src.pa(a + j);
        if (v >= 200.0f) {
            hits++;
            first = min(first, j);
            lastp = j;
            bool gap = true;
            for (int k = 1; k < 10 && gap; k++)
                if (j - k >= 0 && C.src.pa(a + j - k) >= 200.0f) gap = false;
            if (gap) { ncand++; lastc = j; }
        }
    }
    if (hits) {
        atomicAdd(&sh[0], hits);
        atomicMin(&sh[1], first);
        atomicMax(&sh[2], lastp);
    }
    __syncthreads();
    const int tot_hits = sh[0], first_hit = sh[1], last_hit = sh[2];
    int result_n;
    if (tot_hits == 0) {
        result_n = 0;
    } else if (tot_hits == 1) {
        result_n = 1;
        if (tid == 0) rec->open_pores[0] = a + first_hit;
        *last = a + first_hit;
    } else {
        // the first hit is always a "gap" candidate but never reported (the loop starts at i = 1)
        if (first_hit >= j0 && first_hit < j1) { ncand--; if (lastc == first_hit) lastc = -1; }
        // ordered compaction of the reported positions
        int incl = ncand;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int v = __shfl_up_sync(ADB_FULL, incl, o);
            if ((tid & 31) >= o) incl += v;
        }
        __syncthreads();
        if ((tid & 31) == 31) C.S.warp_tot[tid >> 5] = (uint32_t)incl;
        if (lastc >= 0) atomicMax(&sh[4], lastc);
        __syncthreads();
        int wbase = 0, total = 0;
        for (int w = 0; w < (int)((T + 31) >> 5); w++) {
            if (w < (tid >> 5)) wbase += (int)C.S.warp_tot[w];
            total += (int)C.S.warp_tot[w];
        }
        int pos = wbase + incl - ncand;
        if (total > 0) {
            if (ncand > 0 && pos < ADB_MAX_OPEN_PORES) {
                for (int j = j0; j < j1 && pos < ADB_MAX_OPEN_PORES; j++) {
                    if (j == first_hit) continue;
                    if (C.src.pa(a + j) >= 200.0f) {
                        bool gap = true;
                        for (int k = 1; k < 10 && gap; k++)
                            if (j - k >= 0 && C.src.pa(a + j - k) >= 200.0f) gap = false;
                        if (gap) rec->open_pores[pos++] = a + j;
                    }
                }
            }
            result_n = total;
            *last = a + sh[4];
        } else {
            result_n = 1;  // valid_pos = pos[-1]
            if (tid == 0) rec->open_pores[0] = a + last_hit;
            *last = a + last_hit;
        }
    }
    __syncthreads();
    return result_n;
}

struct PrimaryBounds {
    int adapter_start, adapter_end, polya_end;
    int n_topk;           // -1: polya_end_topk is None
    const int *topk;      // n_topk entries (shared or global)
};

// validate_boundaries (combined.py:358-631).  Fills `rec` (thread 0 writes the scalars).  CTA-wide.
__device__ void validate_boundaries_cta(ValCtx &C, const PrimaryBounds &B, int full_len, adb_record *rec) {
    const adb_config &cfg = *C.cfg;
    const int size = C.src.n;
    VcOut o = vc_out(B.adapter_start);
    int a_end = B.adapter_end, pe_best = B.polya_end;
    float a_med = CUDART_NAN_F, a_mad = CUDART_NAN_F;
    bool have_amed = false;
    int mvs_a_end = 0;
    bool polya_none = false;
    const int a_end0 = B.adapter_end;
    float polya_med_cache = 0.f, polya_mad_cache = 0.f; int polya_med_cache_pe = -1;
    bool lr0_ok = false; double lr0 = 0.0;

    if (a_end == 0) {
        o.success = false; o.fail = ADB_FAIL_NO_ADAPTER;
    } else {
        // the local range of real_range_check covers the same samples when the adapter is short and no open
        // pore moves its start: take it from the same histogram
        int ca = o.a_start, cb = a_end;
        clip_seg(ca, cb, size);
        lr0_ok = cfg.real_signal_check && (cb - ca) <= cfg.max_obs_local_range;
        const SegStats A0 = seg_stats(C, o.a_start, a_end, SS_MED | SS_MAD | (lr0_ok ? SS_LR : 0));
        a_med = A0.med; a_mad = A0.mad; lr0 = A0.lr;
        have_amed = true;
    }
    if (o.success && (a_mad != 0.0f) && !in_range_d((double)a_mad, cfg.adapter_mad_range)) {
        o.success = false; o.fail = ADB_FAIL_ADAPTER_MAD;
    }
    const int a_start0 = o.a_start;
    if (o.success && cfg.detect_open_pores) {
        int last = 0;
        o.n_open = open_pores_scan(C, o.a_start, a_end, rec, &last);
        o.valid |= ADB_V_OPEN_PORES;
        if (o.n_open > 0) {
            o.a_start = last;
            if (a_end - o.a_start < cfg.min_obs_adapter) { o.success = false; o.fail = ADB_FAIL_OPEN_PORE; }
        }
    }
    if (o.success && cfg.real_signal_check) {
        int a = o.a_start, b = a_end;
        clip_seg(a, b, size);
        const int len = b - a;
        if (len < 2 * cfg.mean_window) {
            o.success = false; o.fail = ADB_FAIL_REAL_RANGE;
        } else {
            float m0, m1;
            seg_mean_exact_pair(C, a, b - cfg.mean_window, cfg.mean_window, m0, m1);
            o.real[0] = (double)m0; o.real[1] = (double)m1;
            o.valid |= ADB_V_REAL_MEANS;
            if (in_range_d((double)m0, cfg.mean_start_range) && in_range_d((double)m1, cfg.mean_end_range)) {
                const int w = min(cfg.max_obs_local_range, len);
                const double lr = (lr0_ok && o.a_start == a_start0 && w == len) ? lr0 : seg_stats(C, b - w, b, SS_MED | SS_LR).lr;
                o.real[2] = lr;
                o.valid |= ADB_V_REAL_RANGE;
                if (!in_range_d(lr, cfg.local_range)) { o.success = false; o.fail = ADB_FAIL_REAL_RANGE; }
            } else {
                o.success = false; o.fail = ADB_FAIL_REAL_RANGE;
            }
        }
    }
    if (o.success && cfg.mvs_detect_check) {
        if (pe_best == 0) {
            o.success = false; o.fail = ADB_FAIL_NO_POLYA;
        } else {
            double mr[2];
            if (!vc_pa_mean_bounds(cfg, a_med, mr)) { o.exception = true; o.fail = ADB_FAIL_EXC_PA_MEAN_RANGE; }
            else if (B.n_topk < 0) { o.exception = true; o.fail = ADB_FAIL_EXC_TOPK_NONE; }
            const double mlo = mr[0], mhi = mr[1];
            if (!o.exception && cfg.mvs_detect_overwrite) {
                // combined.py:517-566.  The detection only depends on adapter_end, which changes on success only,
                // and success ends the loop: every further candidate after a failure repeats the same evaluation.
                if (B.n_topk > 0 && B.topk[0] != 0) {
                    const bool f64_bounds = cfg.pA_mean_range_empty != 0;
                    const MvsLocOut R = mvs_detect_at_loc(C, a_end, mlo, mhi, f64_bounds);
                    for (int i = 0; i < 5; i++) o.mvs[i] = R.v[i];
                    mvs_a_end = R.idx;
                    o.valid |= ADB_V_MVS | ADB_V_MVS_ADAPTER_END;
                    if (!R.ok) {
                        o.success = false; o.fail = ADB_FAIL_MVS_NO_ADAPTER;
                    } else {
                        int pe = B.topk[0];
                        if (R.idx - a_end > 0) {
                            a_end = R.idx;
                            if (a_end > pe) {
                                // polya_end_adjust and polya_truncated are None in v0.2.4, so polya_end becomes
                                // trace_early_stop_pos -- None as well (combined.py:560-562)
                                polya_none = true;
                                o.valid |= ADB_V_TO_EARLY_STOP | ADB_V_POLYA_NONE;
                            }
                        }
                        pe_best = pe;
                    }
                }
            } else
            if (!o.exception) {
                // combined.py:464-566.  `success` is never set back to True, so once the first candidate fails the
                // reference evaluates EVERY remaining non-zero candidate and ends with: the values of the LAST
                // candidate, the fail reason of the last candidate that failed, polya_end = the first candidate.
                // The checks are pure functions of (adapter_end, candidate), so the same final state follows from
                // candidate 0, then the last candidate, then -- only while those pass -- the ones before it.
                int n_eval = 0;
                while (n_eval < B.n_topk && B.topk[n_eval] != 0) n_eval++;
                if (n_eval > 0) {
                    const int pe0 = B.topk[0];
                    const MvsOut R0 = mvs_check(C, a_end, pe0, mlo, mhi);
                    for (int i = 0; i < 5; i++) o.mvs[i] = R0.v[i];
                    o.valid |= ADB_V_MVS;
                    if (R0.ok || R0.v[0] != 0.0) { polya_med_cache = (float)R0.v[2]; polya_mad_cache = R0.polya_mad; polya_med_cache_pe = pe0; }
                    if (R0.ok) {
                        pe_best = pe0;
                    } else {
                        o.success = false;
                        vc_mvs_fail(R0.v[0], R0.fail_mask, o.fail, o.fail_mask);
                        bool fail_known = false;  // fail reason of the last failing candidate found?
                        for (int t = n_eval - 1; t >= 1 && !fail_known; t--) {
                            const MvsOut R = mvs_check(C, a_end, B.topk[t], mlo, mhi);
                            if (t == n_eval - 1) for (int i = 0; i < 5; i++) o.mvs[i] = R.v[i];
                            if (!R.ok) { vc_mvs_fail(R.v[0], R.fail_mask, o.fail, o.fail_mask); fail_known = true; }
                        }
                    }
                }
            }
        }
    }
    if (!o.exception && o.success && cfg.detect_med_shift) {
        const int w = cfg.med_shift_window;
        const float m_after = seg_stats(C, a_end, min(a_end + w, full_len), SS_MED).med;
        const float m_before = seg_stats(C, max(a_end - w, 0), a_end, SS_MED).med;
        o.med_shift = (double)__fsub_rn(m_after, m_before);
        o.valid |= ADB_V_MED_SHIFT;
        if (!in_range_d(o.med_shift, cfg.med_shift_range)) { o.success = false; o.fail = ADB_FAIL_MED_SHIFT; }
    }
    if (o.exception) {
        if (threadIdx.x == 0) vc_write_exception(rec, o.fail, full_len, size);
        return;
    }
    // partition statistics (signal_partitions.py:65-96), with the updated adapter_start
    const int a_start = o.a_start;
    double st[3][4];
    for (int p = 0; p < 3; p++) for (int q = 0; q < 4; q++) st[p][q] = 0.0;
    if (a_end > a_start) {
        seg_mean_std(C, a_start, a_end, st[0][0], st[0][1]);
        float med = a_med, mad = a_mad;
        if (!(have_amed && a_start == a_start0 && a_end == a_end0)) {
            const SegStats Q = seg_stats(C, a_start, a_end, SS_MED | SS_MAD);
            med = Q.med; mad = Q.mad;
        }
        st[0][2] = (double)med; st[0][3] = (double)mad;
        o.valid |= ADB_V_ADAPTER_STATS;
    }
    if (polya_none) pe_best = 0;  // calc_partition_stats(…, None): no polya and no rna partition
    if (!polya_none && pe_best > a_end) {
        seg_mean_std(C, a_end, pe_best, st[1][0], st[1][1]);
        float med = polya_med_cache, mad = polya_mad_cache;
        if (polya_med_cache_pe != pe_best) {
            const SegStats Q = seg_stats(C, a_end, pe_best, SS_MED | SS_MAD);
            med = Q.med; mad = Q.mad;
        }
        st[1][2] = (double)med; st[1][3] = (double)mad;
        o.valid |= ADB_V_POLYA_STATS;
    }
    if (!polya_none && size > pe_best) {
        seg_mean_std(C, pe_best, size, st[2][0], st[2][1]);
        const SegStats Q = seg_stats(C, pe_best, size, SS_MED | SS_MAD);
        const float med = Q.med, mad = Q.mad;
        st[2][2] = (double)med; st[2][3] = (double)mad;
        o.valid |= ADB_V_RNA_STATS;
    }
    if (threadIdx.x == 0)
        vc_write_record(rec, o, st, full_len, size, a_end, pe_best, B.adapter_end, B.polya_end, mvs_a_end, B.n_topk, B.topk);
}
