// Read-until sessions of the streaming poly(A) detector (SURVEY.md row f4): mean_var_shift_polyA_detect,
// adapted/detect/mvs.py:341-426, asked again every time a channel's cache grows by a chunk.
//
// A session keeps per slot (one per sequencer channel) the cache of the read on it -- int16 ADC codes with the read's
// calibration, or calibrated float32 pA -- and everything the stateless mvs_stream_kernel (adb_stream.cuh) would
// recompute from the start:
//   - the state of the two bottleneck recurrences over signal[min_obs_adapter:] (running sum of the mean; amean /
//     assqdm of the variance; tail samples consumed).  Both are trailing windows evaluated by sequential float32
//     recurrences, so continuing them over the appended samples reproduces the stateless series bit for bit;
//   - the match mask "moving mean and variance in range", which is therefore prefix-stable: only bits for the new
//     positions are appended;
//   - the running min / max sample key (ADC code + 32768, or f32_key of the pA value), which replaces the whole-window
//     scan that bounds the order statistics;
//   - the resume offset of the search loop.  A hit at idx is judged on [idx, idx + polyA_window),
//     [idx, idx + median_shift_window) and [idx - median_shift_window, idx), each clipped at n, and on the
//     n - idx < min_obs_post_loc exit.  Once n - idx >= max(min_obs_post_loc, polyA_window, median_shift_window)
//     no further sample changes that decision, and the hit itself (the first mask bit at or after the offset) is
//     final as soon as it is found.  A final rejection advances the resume offset as the reference advances
//     `offset`; a final acceptance settles the slot.  Decisions on clipped windows are taken again on the next push.
// The early return n < min_obs_adapter + max(windows) is tested on every push.  A slot also settles when its cache
// is full (max_samples): later samples of that read are dropped.
//
// Two launches per push: stream_append_kernel (one warp per pushed slot copies the chunk into the cache and updates
// the key bounds; its lane 0 advances the recurrences and the mask) and stream_search_kernel (one CTA per pushed
// slot resumes the search loop with seg_stats reading the cache in global memory, so a cache is not bounded by
// shared memory).  Float32 sessions run stream_append_f32_kernel / stream_search_f32_kernel: the same code
// (sess_append / sess_search) with the samples taken as they are, and order statistics on float keys through the
// generic multi-level select instead of the one-pass code histogram.
//
// Device pushes (adb_stream_session_push_dev) take entries and chunks in device memory and run on the caller's stream
// with no host synchronise: stream_dev_stamp_kernel and stream_dev_check_kernel validate the whole push and build the
// entries before any state changes, then stream_append_dev_kernel / stream_search_dev_kernel run sess_append /
// sess_search on the caller's buffer unless the push was refused, and write the answers and the status.
#pragma once
#include "adb_stream.cuh"

struct SessSlot {  // device state of one slot
    int32_t n;        // samples in the cache
    int32_t t;        // tail samples (positions >= min_obs_adapter) the recurrences have consumed
    int32_t roff;     // resume offset of the search loop (tail index)
    int32_t result;   // last answer
    int32_t settled;  // the answer is final
    uint32_t kmin, kmax;  // key bounds of the cache (kmin > kmax: empty)
    float coff, cscale;   // calibration of an int16 read (unused by float32 slots)
    float amean, assqdm, asum;
};

struct SessEntry {  // one pushed slot, host -> device (device pushes: built by stream_dev_check_kernel)
    int32_t slot, reset, len, _pad;
    int64_t src;      // first sample of the chunk in the staged blob (device pushes: in the caller's buffer)
    float coff, cscale;
};

template <class T>
struct SessArgsT {
    SessSlot *slots;
    T *cache;              // [n_slots][max_samples]
    uint32_t *mask;        // [n_slots][mask_words]
    const SessEntry *ent;  // [n_ent]
    const T *blob;         // staged chunks
    int32_t *out;          // [n_ent][2]: polya_start, settled
    int n_ent, max_samples, mask_words;
};
struct SessArgs : SessArgsT<int16_t> {};   // int16 ADC caches
struct SessArgsF32 : SessArgsT<float> {};  // calibrated float32 pA caches

// what differs between the two cache types: the order-preserving key of a sample, its pA value, and how seg_stats
// reads the cache
template <class T>
struct SessSample;
template <>
struct SessSample<int16_t> {
    static constexpr bool int_keys = true;  // the session only takes scale > 0
    static __device__ __forceinline__ uint32_t key(int16_t v) { return (uint32_t)((int)v + 32768); }
    static __device__ __forceinline__ float pa(int16_t v, float coff, float cscale) {
        return __fmul_rn(__fadd_rn((float)v, coff), cscale);
    }
    static __device__ __forceinline__ void src(ReadSrc &s, const int16_t *cache) { s.f32 = nullptr; s.i16 = cache; }
};
template <>
struct SessSample<float> {
    static constexpr bool int_keys = false;
    static __device__ __forceinline__ uint32_t key(float v) { return f32_key(v); }
    static __device__ __forceinline__ float pa(float v, float, float) { return v; }
    static __device__ __forceinline__ void src(ReadSrc &s, const float *cache) { s.f32 = cache; s.i16 = nullptr; }
};

#define SESS_APPEND_WARPS 4

// warp of entry e; the kernels compute e and lane, where the compiler knows the bounds of threadIdx.x
template <class T>
__device__ __forceinline__ void sess_append(SessArgsT<T> A, adb_stream_config P, int e, int lane) {
    using X = SessSample<T>;
    if (e >= A.n_ent) return;
    const SessEntry E = A.ent[e];
    SessSlot &S = A.slots[E.slot];
    const int wm = P.pA_mean_window, wv = P.pA_var_window, moa = P.min_obs_adapter;
    if (E.reset) {
        if (lane == 0) {
            S.n = 0; S.t = 0; S.roff = max(wm, wv); S.result = 0; S.settled = 0;
            S.kmin = 0xffffffffu; S.kmax = 0u;
            S.coff = E.coff; S.cscale = E.cscale;
            S.amean = 0.f; S.assqdm = 0.f; S.asum = 0.f;
        }
        __syncwarp();
    }
    if (S.settled || E.len <= 0) return;
    const int n0 = S.n, n1 = n0 + E.len;
    T *cache = A.cache + (size_t)E.slot * A.max_samples;
    uint32_t lo = 0xffffffffu, hi = 0u;
    for (int j = lane; j < E.len; j += 32) {
        const T v = A.blob[E.src + j];
        cache[n0 + j] = v;
        const uint32_t k = X::key(v);
        lo = min(lo, k);
        hi = max(hi, k);
    }
    lo = warp_min_u(lo);
    hi = warp_max_u(hi);
    __syncwarp();  // the chunk is in the cache for lane 0 (warp-level memory ordering)
    if (lane != 0) return;
    S.kmin = min(S.kmin, lo);
    S.kmax = max(S.kmax, hi);
    S.n = n1;
    const int L = n1 - moa;
    int i = S.t;
    if (L <= i) return;
    const float coff = S.coff, cscale = S.cscale;
    auto pa = [&](int j) { return X::pa(cache[j], coff, cscale); };
    float amean = S.amean, assqdm = S.assqdm, asum = S.asum, mv = 0.f, mm = 0.f;
    const float vinv = (float)(1.0 / (double)wv), minv = (float)(1.0 / (double)wm);
    const int i0 = max(wv, wm) - 1;
    uint32_t *mask = A.mask + (size_t)E.slot * A.mask_words;
    uint32_t bits = (i & 31) ? (mask[i >> 5] & ((1u << (i & 31)) - 1u)) : 0u;
    for (; i < L; i++) {
        const float ai = pa(moa + i);
        if (i < wv) {
            mv_var_warm(amean, assqdm, ai, i);
            if (i == wv - 1) mv = mv_var_first(assqdm, wv);
        } else {
            mv_var_step(amean, assqdm, ai, pa(moa + i - wv), vinv);
            mv = __fmul_rn(assqdm, vinv);
        }
        if (i < wm) {
            asum = __fadd_rn(asum, ai);
            if (i == wm - 1) mm = __fdiv_rn(asum, (float)wm);
        } else {
            asum = mv_mean_step(asum, ai, pa(moa + i - wm));
            mm = __fmul_rn(asum, minv);
        }
        if (i >= i0 && in_range_f32w(mm, P.pA_mean_range) && in_range_f32w(mv, P.pA_var_range)) bits |= 1u << (i & 31);
        if ((i & 31) == 31) { mask[i >> 5] = bits; bits = 0u; }
    }
    if (L & 31) mask[L >> 5] = bits;
    S.t = L;
    S.amean = amean; S.assqdm = assqdm; S.asum = asum;
}

__global__ void __launch_bounds__(SESS_APPEND_WARPS * 32) stream_append_kernel(SessArgs A, adb_stream_config P) {
    sess_append(A, P, blockIdx.x * SESS_APPEND_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}
__global__ void __launch_bounds__(SESS_APPEND_WARPS * 32) stream_append_f32_kernel(SessArgsF32 A, adb_stream_config P) {
    sess_append(A, P, blockIdx.x * SESS_APPEND_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

template <class T>
__device__ __forceinline__ void sess_search(SessArgsT<T> A, adb_stream_config P) {
    using X = SessSample<T>;
    __shared__ __align__(16) unsigned char scratch[((size_t)ADB_SEL_SMEM_BYTES + 64 + 15) & ~(size_t)15];
    __shared__ uint32_t kbuf[8];
    __shared__ int itmp[8];
    __shared__ double dtmp[8];
    const int e = blockIdx.x;
    const SessEntry E = A.ent[e];
    SessSlot &S = A.slots[E.slot];
    if (S.settled) {
        if (threadIdx.x == 0) { A.out[2 * e] = S.result; A.out[2 * e + 1] = 1; }
        return;
    }
    const int wm = P.pA_mean_window, wv = P.pA_var_window, moa = P.min_obs_adapter;
    const int n = S.n;
    const bool full = n >= A.max_samples;
    int result = 0, settled = full ? 1 : 0, roff = S.roff;
    if (n >= moa + max(max(wm, wv), max(P.min_obs_post_loc, P.polyA_window))) {  // mvs.py:352-363
        ValCtx C;
        C.cfg = nullptr;
        C.S = sel_scratch_from(scratch);
        C.kbuf = kbuf;
        C.itmp = itmp;
        C.dtmp = dtmp;
        C.series_a = C.series_b = nullptr;
        C.pre_var = C.pre_mean = nullptr;
        C.pre_ae = C.pre_pe = -1;
        X::src(C.src, A.cache + (size_t)E.slot * A.max_samples);
        C.src.n = n;
        C.src.coff = S.coff;
        C.src.cscale = S.cscale;
        C.int_keys = X::int_keys;
        C.wkmin = S.kmin;
        C.wkmax = S.kmax;
        const PaVal V{C.src, X::int_keys};
        C.wvmin = V(C.wkmin);
        C.wvmax = V(C.wkmax);
        const uint32_t *mask = A.mask + (size_t)E.slot * A.mask_words;
        const int L = n - moa, nwords = (L + 31) >> 5;
        const int need = max(P.min_obs_post_loc, max(P.polyA_window, P.median_shift_window));
        int offset = roff;
        while (offset < L) {  // mvs.py:381-425 from the first decision that was not final
            if (threadIdx.x == 0) itmp[7] = 0x7fffffff;
            __syncthreads();
            for (int w = (offset >> 5) + threadIdx.x; w < nwords; w += blockDim.x) {
                uint32_t bits = mask[w];
                if (w == (offset >> 5)) bits &= 0xffffffffu << (offset & 31);
                if (w == nwords - 1 && (L & 31)) bits &= (1u << (L & 31)) - 1u;  // the word holds no later bit
                if (bits) { atomicMin(&itmp[7], w * 32 + __ffs(bits) - 1); break; }
            }
            __syncthreads();
            const int hit = itmp[7];
            __syncthreads();
            if (hit == 0x7fffffff) break;                     // no match yet
            const int idx = moa + hit;
            if (n - idx < P.min_obs_post_loc) break;          // not enough signal after the hit yet
            const bool final_ = n - idx >= need;
            const SegStats Q = seg_stats(C, idx, min(idx + P.polyA_window, n), SS_MED | SS_LR);
            const float m_after = seg_stats(C, idx, min(idx + P.median_shift_window, n), SS_MED).med;
            const float m_before = seg_stats(C, max(idx - P.median_shift_window, 0), idx, SS_MED).med;
            const double shift = (double)__fsub_rn(m_after, m_before);
            if (in_range_f32w(Q.med, P.polyA_med_range) && in_range_d(Q.lr, P.polyA_local_range) &&
                in_range_d(shift, P.median_shift_range)) {
                result = idx;
                if (final_) settled = 1;
                break;
            }
            offset = idx - moa + P.search_increment_step;
            if (final_) roff = offset;  // every earlier decision was final too: resume here next time
        }
    }
    if (threadIdx.x == 0) {
        S.roff = roff;
        S.result = result;
        S.settled = settled;
        A.out[2 * e] = result;
        A.out[2 * e + 1] = settled;
    }
}

__global__ void __launch_bounds__(ADB_VAL_THREADS) stream_search_kernel(SessArgs A, adb_stream_config P) { sess_search(A, P); }
__global__ void __launch_bounds__(ADB_VAL_THREADS) stream_search_f32_kernel(SessArgsF32 A, adb_stream_config P) {
    sess_search(A, P);
}

// ---- device pushes ----------------------------------------------------------------------------------------------
// Refusals of a push, in the order the host push (session_push, adb_api.cu) checks them.  A refusal is recorded as the
// key (phase << 40) | (entry << 8) | reason and the push keeps the smallest key, so the device reports the refusal the
// host push would report first: the phase orders the host's passes, the entry its per-entry loop.
enum SessReason : int32_t {
    SESS_R_NONE = 0,
    SESS_R_NEG_OFFSET,    // phase 0
    SESS_R_DECREASING,    // phase 1, per entry
    SESS_R_NULL_ADC,      // phase 2
    SESS_R_NULL_PA,       // phase 2
    SESS_R_SLOT_RANGE,    // phase 3, per entry, in this order
    SESS_R_DUPLICATE,
    SESS_R_NO_CALIB,
    SESS_R_BAD_CALIB,
    SESS_R_NOT_STARTED,
    SESS_R_NON_FINITE,    // phase 4
    SESS_R_COUNT
};
#define SESS_DEV_OK 0xffffffffffffffffull
#define SESS_DEV_THREADS 256

struct SessPush {  // the caller's arrays of one device push (device pointers)
    const int32_t *slots;     // [n]
    const int64_t *offs;      // [n + 1] chunk offsets into `samples`
    const void *samples;      // int16 ADC or float32 pA, as the session holds
    const uint8_t *reset;     // [n] or null
    const float *coff, *cscale;  // [n] or null (int16 only)
    int32_t *polya_start;     // [n]
    uint8_t *settled;         // [n]
    int32_t *status;          // [2]: adb_status, SessReason
    int n;
};

struct SessDev {  // state of a device-push session next to SessSlot, and the scratch of one push
    uint32_t *stamp;    // [n_slots] first entry of the running push that names the slot; 0xffffffff between pushes
    uint8_t *started;   // [n_slots] a read was started on the slot by an accepted push
    SessEntry *ent;     // [n_slots] entries of the running push
    unsigned long long *err;  // smallest refusal key of the running push, SESS_DEV_OK if none
    int n_slots;
};

__device__ __forceinline__ void sess_refuse(SessDev D, int phase, int k, int reason) {
    atomicMin(D.err, ((unsigned long long)phase << 40) | ((unsigned long long)(uint32_t)k << 8) | (unsigned)reason);
}
__device__ __forceinline__ bool non_finite_f32(float v) { return (__float_as_uint(v) & 0x7f800000u) == 0x7f800000u; }

// opens the push: clears its refusal key and stamps every slot named with the first entry naming it
__global__ void __launch_bounds__(SESS_DEV_THREADS) stream_dev_stamp_kernel(SessPush Q, SessDev D) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *D.err = SESS_DEV_OK;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < Q.n; k += gridDim.x * blockDim.x) {
        const int sl = Q.slots[k];
        if (sl >= 0 && sl < D.n_slots) atomicMin(&D.stamp[sl], (uint32_t)k);
    }
}

// Every check of the host push, and the entries from device state: entry k appends chunk k straight from the
// caller's buffer (src = chunk_offsets[k]), clipped at max_samples; a settled slot that is not reset gets a
// zero-length entry, for which sess_search returns the final answer.  Float32 sessions also scan every sample of
// [chunk_offsets[0], chunk_offsets[n]) for NaN / inf, chunks of settled slots and clipped samples included.
template <class T>
__device__ __forceinline__ void sess_dev_check(SessArgsT<T> A, SessPush Q, SessDev D) {
    constexpr bool f32 = !SessSample<T>::int_keys;
    const int stride = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t o0 = Q.offs[0], o1 = Q.offs[Q.n];
    if (tid == 0) {
        if (o0 < 0) sess_refuse(D, 0, 0, SESS_R_NEG_OFFSET);
        if (o1 > o0 && !Q.samples) sess_refuse(D, 2, 0, f32 ? SESS_R_NULL_PA : SESS_R_NULL_ADC);
    }
    for (int k = tid; k < Q.n; k += stride) {
        const int64_t a = Q.offs[k], b = Q.offs[k + 1];
        if (b < a) sess_refuse(D, 1, k, SESS_R_DECREASING);
        const int sl = Q.slots[k];
        const bool rs = Q.reset && Q.reset[k];
        int r = SESS_R_NONE;
        if (sl < 0 || sl >= D.n_slots) {
            r = SESS_R_SLOT_RANGE;
        } else if (D.stamp[sl] != (uint32_t)k) {  // reads k' < k, or the cleared stamp once entry k' is through
            r = SESS_R_DUPLICATE;
        } else {
            D.stamp[sl] = 0xffffffffu;
            if (rs) {
                if (!f32) {
                    if (!Q.coff || !Q.cscale) r = SESS_R_NO_CALIB;
                    else if (!isfinite(Q.cscale[k]) || !(Q.cscale[k] > 0.f) || !isfinite(Q.coff[k])) r = SESS_R_BAD_CALIB;
                }
            } else if (!D.started[sl]) {
                r = SESS_R_NOT_STARTED;
            }
        }
        if (r != SESS_R_NONE) { sess_refuse(D, 3, k, r); continue; }
        const SessSlot &S = A.slots[sl];
        SessEntry E;
        E.slot = sl;
        E.reset = rs ? 1 : 0;
        E._pad = 0;
        E.src = a;
        E.len = !rs && S.settled ? 0 : (int32_t)min(b - a, (int64_t)(A.max_samples - (rs ? 0 : S.n)));
        E.coff = rs && !f32 ? Q.coff[k] : 0.f;
        E.cscale = rs && !f32 ? Q.cscale[k] : 0.f;
        D.ent[k] = E;
    }
    if (f32 && Q.samples && o0 >= 0 && o1 > o0) {  // block-uniform
        const float *x = (const float *)Q.samples + o0;
        const int64_t cnt = o1 - o0;
        const int64_t head = min(cnt, (int64_t)(((16u - ((uint32_t)(uintptr_t)x & 15u)) & 15u) >> 2));
        const int64_t nv = (cnt - head) >> 2;
        const float4 *v = (const float4 *)(x + head);
        bool bad = false;
        for (int64_t j = tid; j < head; j += stride) bad |= non_finite_f32(x[j]);
        for (int64_t j = tid; j < nv; j += stride) {
            const float4 q = __ldg(v + j);
            bad |= non_finite_f32(q.x) | non_finite_f32(q.y) | non_finite_f32(q.z) | non_finite_f32(q.w);
        }
        for (int64_t j = head + 4 * nv + tid; j < cnt; j += stride) bad |= non_finite_f32(x[j]);
        if (__syncthreads_or(bad) && threadIdx.x == 0) sess_refuse(D, 4, 0, SESS_R_NON_FINITE);
    }
}

__global__ void __launch_bounds__(SESS_DEV_THREADS) stream_dev_check_kernel(SessArgs A, SessPush Q, SessDev D) {
    sess_dev_check(A, Q, D);
}
__global__ void __launch_bounds__(SESS_DEV_THREADS) stream_dev_check_f32_kernel(SessArgsF32 A, SessPush Q, SessDev D) {
    sess_dev_check(A, Q, D);
}

template <class T>
__device__ __forceinline__ void sess_append_dev(SessArgsT<T> A, adb_stream_config P, SessDev D, int e, int lane) {
    if (*D.err != SESS_DEV_OK) return;  // refused: nothing changes
    if (lane == 0 && e < A.n_ent && A.ent[e].reset) D.started[A.ent[e].slot] = 1;
    sess_append(A, P, e, lane);
}
__global__ void __launch_bounds__(SESS_APPEND_WARPS * 32) stream_append_dev_kernel(SessArgs A, adb_stream_config P, SessDev D) {
    sess_append_dev(A, P, D, blockIdx.x * SESS_APPEND_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}
__global__ void __launch_bounds__(SESS_APPEND_WARPS * 32) stream_append_dev_f32_kernel(SessArgsF32 A, adb_stream_config P,
                                                                                      SessDev D) {
    sess_append_dev(A, P, D, blockIdx.x * SESS_APPEND_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// closes the push: the status always, the answers only for an accepted push (a refused one leaves them untouched)
template <class T>
__device__ __forceinline__ void sess_search_dev(SessArgsT<T> A, adb_stream_config P, SessDev D, SessPush Q) {
    const unsigned long long err = *D.err;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        Q.status[0] = err == SESS_DEV_OK ? ADB_OK : ADB_ERR_ARG;
        Q.status[1] = err == SESS_DEV_OK ? SESS_R_NONE : (int32_t)(err & 0xffu);
    }
    if (err != SESS_DEV_OK) return;
    sess_search(A, P);
    if (threadIdx.x == 0) {  // sess_search wrote them from this thread
        Q.polya_start[blockIdx.x] = A.out[2 * blockIdx.x];
        Q.settled[blockIdx.x] = A.out[2 * blockIdx.x + 1] ? 1 : 0;
    }
}
__global__ void __launch_bounds__(ADB_VAL_THREADS) stream_search_dev_kernel(SessArgs A, adb_stream_config P, SessDev D,
                                                                            SessPush Q) {
    sess_search_dev(A, P, D, Q);
}
__global__ void __launch_bounds__(ADB_VAL_THREADS) stream_search_dev_f32_kernel(SessArgsF32 A, adb_stream_config P,
                                                                                SessDev D, SessPush Q) {
    sess_search_dev(A, P, D, Q);
}
