// validate_boundaries + per-segment statistics for int16 sources from HISTOGRAMS BUILT ON THE TENSOR CORES.
//
// Reference: adapted/detect/combined.py:358-631 (the checks and the record: adb_vcheck.cuh, shared with adb_vfast.cuh).
//
// Every order statistic the reference asks for (medians, MADs, p15 / p85 of up to a dozen sample ranges of a read) is
// a function of the histogram of the ADC codes of the range.  Shared-memory atomics build such a histogram at 2 cycles
// per sample and SM (profiles/r1_validate_kernel_v3.txt), counting passes need ~20 passes over the window
// (adb_vfast.cuh).  Here the tensor core does the scatter-add: for 32 consecutive samples a warp writes two ONE-HOT
// operand tiles in shared memory,
//     A[hi][k] = 1 iff (code_k - base) >> 4 == hi      (M = 64 rows)
//     B[lo][k] = 1 iff (code_k - base) & 15 == lo      (N = 16 rows)
// (one byte store per sample and tile, e4m3 1.0 = 0x38) and one tcgen05.mma.kind::f8f6f4 (K = 32) accumulates
//     D[hi][lo] += sum_k A[hi][k] * B[lo][k]  =  number of samples of the batch with code - base == 16 * hi + lo
// into a float32 accumulator in TMEM (exact: counts stay below 2^24) -- a 1024-bin histogram per accumulator, no
// atomics, no conflicts between samples of equal value.  A warp batch is 64 samples (two MMAs, one fence, one commit);
// after the MMAs have read the tiles the warp clears the bytes it set (the tiles are all-zero between batches).  The
// tensor core reads the whole (mostly zero) tiles: 80 B of shared memory per sample -- the floor of this formulation
// (M >= 64 for tcgen05), reached by the stream phase.
//
// The ranges of a read overlap (adapter, its tail windows, poly(A), the windows around adapter_end, the rest), so the
// window is cut at every range boundary into at most VH_MAX_PIECES disjoint PIECES, one accumulator each (16 TMEM
// columns, 128 columns per CTA, four CTAs per SM); a range is a run of consecutive pieces.  The samples are read ONCE
// from global memory (no staging of the window in shared memory; the next read's window is prefetched into L2), the
// exact sums of the codes and of their squares per piece are taken on the way.  The accumulators are then copied to
// shared memory as per-piece cumulative counts and every statistic is a few look-ups in them: ranks by 32-way searches
// (one warp per query), MADs by 32-way searches for the first candidate deviation whose count exceeds the middle rank
// (the two sides of a median on two warps), with exact float32 deviations.  The checks and the record run on warp 0.
//
// Codes outside [base, base + 1023] (base = the code of 25 pA: the range covers 25 .. 205 pA at a typical calibration)
// fall into the end bins; a read is handed to validate_kernel (same results) whenever an answer or a decisive probe
// touches an end bin that holds such codes.  Also handed over: what validate_fast_kernel hands over (the same checks).
#pragma once
#include "adb_cnn_tc.cuh"
#include "adb_vfast.cuh"

#define VH_M 64                            // rows of the A tile = values of the high part of a code offset
#define VH_BINS (VH_M * 16)
#define VH_MAX_PIECES 8
#define VH_A_LBO (VH_M * 16 + 64)          // A tile: 2 K-groups (16 samples each) of VH_M rows x 16 B, 64 B apart in banks
#define VH_A_BYTES (VH_A_LBO + VH_M * 16)
#define VH_B_LBO 320                       // B tile: 2 K-groups of 16 rows x 16 B
#define VH_B_BYTES (VH_B_LBO + 256)
#define VH_TILE_BYTES ((VH_A_BYTES + VH_B_BYTES + 127) & ~127)  // A + B of one warp
#define VH_WARPS (VF_THREADS / 32)
#define VH_SUB 2                           // MMAs (32 samples each) per batch of a warp: one fence, commit and wait for both
#define VH_ARENA_TILES (VH_WARPS * VH_SUB * VH_TILE_BYTES)
#define VH_ARENA_CUM (VH_MAX_PIECES * VH_BINS * 2)   // cumulative counts, u16
#define VH_ARENA (VH_ARENA_TILES > VH_ARENA_CUM ? VH_ARENA_TILES : VH_ARENA_CUM)
// instruction descriptor: D = f32, A = B = e4m3 (0), K-major, N = 16, M = VH_M
#define VH_IDESC ((1u << 4) | ((16u >> 3) << 17) | (((unsigned)VH_M >> 4) << 24))
#define VH_OP_WORDS 512                    // open-pore scan: 16 384 samples of adapter at most

#ifdef ADB_VH_STATS
__device__ unsigned long long vh_dbg[16];  // [0] reads, [1..] cycles of the phases (thread 0)
#define VH_T(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(&vh_dbg[i], (unsigned long long)(t_ - vh_t0)); vh_t0 = t_; } } while (0)
#else
#define VH_T(i) do { } while (0)
#endif

__host__ __device__ inline size_t vhist_smem_bytes() { return (size_t)VH_ARENA + 128; }

__device__ __forceinline__ void vh_mma_f8(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], da, db, %5, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(VH_IDESC)
        : "memory");
}

__device__ __forceinline__ void vh_tmem_zero32(uint32_t taddr) {
    const uint32_t z = 0u;
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
        "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};\n" ::"r"(taddr),
        "r"(z)
        : "memory");
}

__device__ __forceinline__ void vh_tmem_ld16(uint32_t taddr, uint32_t v[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct VhShared {
    VfScratch S;                       // scratch of the helpers shared with adb_vfast.cuh
    uint64_t bar[VH_WARPS];            // "the MMAs of this warp's batch have read the tiles"
    uint32_t tmem_slot;
    int cuts[VH_MAX_PIECES + 4];       // sorted cut points; piece p = samples [cuts[p], cuts[p + 1])
    int np;
    int n_low, n_high;                 // samples of the read below base / above base + 2047
    int unsettled;                     // an answer or a probe touched an end bin holding such samples
    VcIn in;                           // the read's inputs, for the checks (kept out of registers through the pass)
    int mfp[4][2];                     // first passing candidate of the right / left side of the four MAD ranges
    uint32_t hitw[VH_OP_WORDS];        // vh_open_pores: bit i = sample i of the aligned window is an open-pore sample
    unsigned long long psum[VH_MAX_PIECES][2];  // per piece: sum of (code - base), sum of (code - base)^2 (exact)
};

// samples of the pieces [p0, p1) whose clamped code offset is <= x
__device__ __forceinline__ int vh_cle(const uint16_t *cum, int p0, int p1, int x) {
    if (x < 0) return 0;
    x = min(x, VH_BINS - 1);
    int c = 0;
    for (int p = p0; p < p1; p++) c += (int)cum[p * VH_BINS + x];
    return c;
}
// smallest offset x with vh_cle(x) > k (0 <= k < samples of the range).  Warp-cooperative (all lanes, same arguments,
// same result): a 32-way search, three rounds of one look-up per lane instead of eleven dependent ones.
__device__ __forceinline__ int vh_wselect(const uint16_t *cum, int p0, int p1, int k) {
    const int lane = threadIdx.x & 31;
    constexpr int B1 = VH_BINS / 32;                   // bins per first-level block
    unsigned m = __ballot_sync(ADB_FULL, vh_cle(cum, p0, p1, B1 * lane + B1 - 1) > k);
    const int l1 = __ffs(m) - 1;                       // the block holding the answer (bit 31 is always set)
    if (B1 == 32) {
        m = __ballot_sync(ADB_FULL, vh_cle(cum, p0, p1, B1 * l1 + lane) > k);
        return B1 * l1 + __ffs(m) - 1;
    }
    m = __ballot_sync(ADB_FULL, vh_cle(cum, p0, p1, B1 * l1 + 2 * lane + 1) > k);
    const int x = B1 * l1 + 2 * (__ffs(m) - 1);
    return (vh_cle(cum, p0, p1, x) > k) ? x : x + 1;
}

struct VhRange { int p0, p1; };  // pieces of a sample range
__device__ __forceinline__ VhRange vh_range(const VhShared &H, int a, int b, int size) {
    clip_seg(a, b, size);
    VhRange q{0, 0};
    if (b <= a) return q;
    const int np = H.np;
    for (int i = 0; i <= np; i++) {
        if (H.cuts[i] == a) q.p0 = i;
        if (H.cuts[i] == b) q.p1 = i;
    }
    return q;
}

// median(|x - med|) of a range from the cumulative counts.  Warp-cooperative (uniform arguments and results).
// The candidates are the deviations of the codes on either side of the median (right: pv + i, left: pv - 1 - i, both
// non-decreasing in i); d0 = the smallest candidate t with #(deviation <= t) > k.  "Candidate i of a side passes" is
// monotone in i, so each side is a 32-way search for its first passing candidate (one candidate per lane and round:
// exact float32 deviation, the matching end of the interval on the other side, two look-ups) -- the two sides of a range
// run on two warps -- and d0 is the smaller of the two.  The decisive evaluations (first passing, last failing) are
// repeated with the end-bin check.  Candidates are all codes of the histogram range (codes nobody holds are harmless:
// the count only changes at codes that are held, so the first passing candidate of the side that decides is a held one).
struct VhMad {
    const VfRead &R;
    VhShared &H;
    const uint16_t *cum;
    VhRange q;
    int base, n, k, pv, nR, nL, n_low, n_high;
    float med, rscale;
    __device__ VhMad(const VfRead &R_, VhShared &H_, const uint16_t *cum_, VhRange q_, int base_, int n_, float med_)
        : R(R_), H(H_), cum(cum_), q(q_), base(base_), n(n_), med(med_) {
        n_low = H.n_low; n_high = H.n_high;
        k = (n - 1) / 2;
        rscale = 1.0f / R.cscale;
        int ok = 1;
        pv = gsb_code_at(med, false, R.coff, R.cscale, &ok);
        pv = min(max(pv, base), base + VH_BINS);
        nR = base + VH_BINS - pv;
        nL = pv - base;
    }
    __device__ __forceinline__ float sdev(bool right, int i) const { return vf_dev(R, right ? pv + i : pv - 1 - i, med); }
    // first index of a side whose deviation is > thr (strict) or >= thr
    __device__ int sfirst(bool right, int nn, float thr, bool strict) const {
        float gf = thr * rscale;  // (a guess: corrected below by evaluating the deviations exactly)
        int g = (gf == gf && gf < 1e9f) ? (int)gf : nn;
        g = min(max(g, 0), nn);
        int guard = 0;
        while (g > 0 && guard++ < 100000) {
            const float d = sdev(right, g - 1);
            if (strict ? (d > thr) : (d >= thr)) g--; else break;
        }
        while (g < nn && guard++ < 100000) {
            const float d = sdev(right, g);
            if (strict ? !(d > thr) : !(d >= thr)) g++; else break;
        }
        return g;
    }
    // samples deviating at most thr (check: flag the read if the interval runs into an end bin that holds outside codes)
    __device__ int count_le(float thr, bool check) const {
        const int jR = sfirst(true, nR, thr, true), jL = sfirst(false, nL, thr, true);
        const int pA = pv - jL, pB = pv + jR - 1;
        if (pB < pA) return 0;
        const int xa = pA - base, xb = pB - base;
        if (check && ((xa <= 0 && n_low > 0) || (xb >= VH_BINS - 1 && n_high > 0))) H.unsettled = 1;
        return vh_cle(cum, q.p0, q.p1, xb) - vh_cle(cum, q.p0, q.p1, xa - 1);
    }
    // first passing candidate of a side (its number of candidates if none)
    __device__ int first_pass(bool right) const {
        const int lane = threadIdx.x & 31;
        const int nn = right ? nR : nL;
        int lo = 0, hi = nn;
        while (lo < hi) {
            const int step = (hi - lo + 31) >> 5;
            const int i = lo + (lane + 1) * step - 1;     // lanes probe lo + step - 1, lo + 2 step - 1, ...
            const bool pass = (i >= hi) || (count_le(sdev(right, min(i, nn - 1)), false) > k);
            const unsigned m = __ballot_sync(ADB_FULL, pass);  // monotone in the lane
            if (!m) { lo = hi; break; }                        // every candidate probed fails (the last probe was hi - 1)
            const int f = __ffs(m) - 1;
            // the answer lies in (lo + f step - 1, lo + (f + 1) step - 1]
            const int nlo = lo + f * step, nhi = min(lo + (f + 1) * step - 1, hi);
            lo = nlo; hi = nhi;
        }
        return lo;
    }
    __device__ float finish(int fR, int fL) const {
        const int lane = threadIdx.x & 31;
        float d0 = CUDART_INF_F;
        if (fR < nR) d0 = fminf(d0, sdev(true, fR));
        if (fL < nL) d0 = fminf(d0, sdev(false, fL));
        // decisive evaluations with the end-bin check (lanes 0..3), and the count at d0
        {
            const bool right = lane < 2;
            const int f = right ? fR : fL, nn = right ? nR : nL;
            const int i = (lane & 1) ? f - 1 : f;
            if (lane < 4 && i >= 0 && i < nn) (void)count_le(sdev(right, i), true);
        }
        const int c_best = count_le(d0, true);
        if (n & 1) return d0;
        float d1 = d0;
        if (!(c_best > k + 1)) {
            // the next larger deviation: the first occupied code on either side of the interval [l, r] deviating <= d0
            int lo = base, hi = pv;
            while (lo < hi) { const int m = (lo + hi) >> 1; if (vf_dev(R, m, med) <= d0) hi = m; else lo = m + 1; }
            const int l = lo;
            lo = pv; hi = base + VH_BINS;
            while (lo < hi) { const int m = (lo + hi) >> 1; if (vf_dev(R, m, med) > d0) hi = m; else lo = m + 1; }
            const int r = lo - 1;
            d1 = CUDART_INF_F;
            auto touch = [&](int x) { if ((x <= 0 && n_low > 0) || (x >= VH_BINS - 1 && n_high > 0)) H.unsettled = 1; };
            const int c_r = vh_cle(cum, q.p0, q.p1, r - base);          // samples with a code <= r
            if (c_r < n) { const int x = vh_wselect(cum, q.p0, q.p1, c_r); touch(x); d1 = fminf(d1, vf_dev(R, x + base, med)); }
            const int c_l = vh_cle(cum, q.p0, q.p1, l - 1 - base);      // samples with a code < l
            if (c_l > 0) { const int x = vh_wselect(cum, q.p0, q.p1, c_l - 1); touch(x); d1 = fminf(d1, vf_dev(R, x + base, med)); }
        }
        return __fdiv_rn(__fadd_rn(d0, d1), 2.0f);
    }
};

// find_open_pores (anomalies.py:15-35) over the samples [0, b) of the window (b <= 32 * VH_OP_WORDS - 8), any int16
// code.  Same results as vf_open_pores (adb_vfast.cuh), which scans per-thread chunks sample by sample; here the window
// is read once with 16-byte loads into a bit mask (sample is an open-pore sample iff code >= c200) and everything else
// is word arithmetic on the mask: a hit is a run start iff none of the 9 samples before it is a hit.
__device__ int vh_open_pores(const VfRead &R, VhShared &H, int b, int c200, adb_record *rec, int *last) {
    const int tid = threadIdx.x, lane = tid & 31;
    VfScratch &S = H.S;
    int *sh = S.itmp;  // [0] hits, [1] first hit, [2] last hit, [3] run starts (the first hit excluded), [4] last run start
    __syncthreads();
    if (tid == 0) { sh[0] = 0; sh[1] = 0x7fffffff; sh[2] = -1; sh[3] = 0; sh[4] = -1; }
    const int i0 = R.s0, i1 = R.s0 + b;               // aligned-window indices of the samples
    const int nvec = (i1 + 7) >> 3, nwords = (nvec + 3) >> 2;
    const uint4 *V = reinterpret_cast<const uint4 *>(R.W16);
    uint8_t *hb = reinterpret_cast<uint8_t *>(H.hitw);
    for (int v = tid; v < nwords * 4; v += VF_THREADS) {
        unsigned m = 0;
        if (v < nvec) {
            uint4 q = make_uint4(0, 0, 0, 0);
            if ((v << 3) >= R.s0 && ((v + 1) << 3) <= R.s0 + R.n) q = __ldg(V + v);
            else {  // the vector reaches beyond the read (before its first or past its last sample): sample by sample
                unsigned short e[8];
#pragma unroll
                for (int t = 0; t < 8; t++) {
                    const int ii = (v << 3) + t;
                    e[t] = (ii >= R.s0 && ii < R.s0 + R.n) ? R.W16[ii] : (unsigned short)0x8000;
                }
                q = make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
            }
            const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                m |= ((int)(int16_t)(w[t] & 0xffffu) >= c200 ? 1u : 0u) << (2 * t);
                m |= ((int)(int16_t)(w[t] >> 16) >= c200 ? 1u : 0u) << (2 * t + 1);
            }
            const int ib = v << 3;                    // bits outside [i0, i1) off
            if (ib < i0) m &= 0xffu << min(i0 - ib, 8);
            if (ib + 8 > i1) m &= 0xffu >> min(ib + 8 - i1, 8);
        }
        hb[v] = (uint8_t)m;
    }
    __syncthreads();
    // per word: hits, run starts
    int hits = 0, first = 0x7fffffff, lastp = -1;
    for (int w = tid; w < nwords; w += VF_THREADS) {
        const uint32_t h = H.hitw[w];
        if (h) { hits += __popc(h); first = min(first, 32 * w + __ffs(h) - 1); lastp = max(lastp, 32 * w + 31 - __clz(h)); }
    }
    hits = __reduce_add_sync(ADB_FULL, hits);
    first = __reduce_min_sync(ADB_FULL, first);
    lastp = __reduce_max_sync(ADB_FULL, lastp);
    if (lane == 0 && hits) { atomicAdd(&sh[0], hits); atomicMin(&sh[1], first); atomicMax(&sh[2], lastp); }
    __syncthreads();
    const int tot_hits = sh[0], first_hit = sh[1], last_hit = sh[2];  // (aligned-window indices)
    int result_n = 0;
    if (tot_hits == 1) {
        result_n = 1;
        if (tid == 0) rec->open_pores[0] = first_hit - i0;
        *last = first_hit - i0;
    } else if (tot_hits > 1) {
        // run starts other than the first hit, in order: counted per word, placed by a prefix sum over the words
        // (nwords <= 512 = two words per thread)
        uint32_t c[2] = {0, 0};
        int n2 = 0;
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int w = 2 * tid + u;
            if (w < nwords) {
                const uint32_t h = H.hitw[w], pv = w ? H.hitw[w - 1] : 0u;
                uint32_t near = 0;
#pragma unroll
                for (int k = 1; k <= 9; k++) near |= (h << k) | (pv >> (32 - k));
                c[u] = h & ~near;
                if ((first_hit >> 5) == w) c[u] &= ~(1u << (first_hit & 31));
                n2 += __popc(c[u]);
            }
        }
        int incl = n2;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(ADB_FULL, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) S.wtot[tid >> 5] = (unsigned)incl;
        int lastc = -1;
        if (c[1]) lastc = 32 * (2 * tid + 1) + 31 - __clz(c[1]); else if (c[0]) lastc = 32 * (2 * tid) + 31 - __clz(c[0]);
        lastc = __reduce_max_sync(ADB_FULL, lastc);
        if (lane == 0 && lastc >= 0) atomicMax(&sh[4], lastc);
        __syncthreads();
        int wbase = 0, total = 0;
        for (int q = 0; q < VF_THREADS / 32; q++) { if (q < (tid >> 5)) wbase += (int)S.wtot[q]; total += (int)S.wtot[q]; }
        if (total > 0) {
            int pos = wbase + incl - n2;
#pragma unroll
            for (int u = 0; u < 2; u++) {
                uint32_t m = c[u];
                while (m && pos < ADB_MAX_OPEN_PORES) {
                    const int bit = __ffs(m) - 1;
                    m &= m - 1;
                    rec->open_pores[pos++] = 32 * (2 * tid + u) + bit - i0;
                }
            }
            result_n = total;
            *last = sh[4] - i0;
        } else {
            result_n = 1;
            if (tid == 0) rec->open_pores[0] = last_hit - i0;
            *last = last_hit - i0;
        }
    }
    __syncthreads();
    return result_n;
}

__global__ void __launch_bounds__(VF_THREADS, 4) validate_hist_kernel(VfastArgs A, adb_config cfg) {
    extern __shared__ __align__(128) unsigned char vh_smem[];
    unsigned char *arena = vh_smem;                                   // operand tiles, later the cumulative counts
    uint16_t *cum = reinterpret_cast<uint16_t *>(arena);
    __shared__ VhShared H;
    VfScratch &S = H.S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int w = 0; w < VH_WARPS; w++) mbar_init(&H.bar[w], 1);
    }
    for (int i = tid; i < VH_ARENA / 16; i += VF_THREADS) reinterpret_cast<uint4 *>(arena)[i] = make_uint4(0, 0, 0, 0);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(&H.tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = H.tmem_slot;
    {
        const uint32_t t0 = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(warp >> 2) * 64;
        vh_tmem_zero32(t0);
        vh_tmem_zero32(t0 + 32);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    unsigned char *tile0 = arena + (size_t)warp * VH_SUB * VH_TILE_BYTES;
    const uint32_t ab_hi = tc_desc_hi(128);
    // descriptors of sub-tile 0 (sub-tile u: + u * VH_TILE_BYTES >> 4 in the address field); this lane's byte of a tile row
    const uint32_t a_lo0 = tc_desc_lo(smem_u32(tile0), VH_A_LBO), b_lo0 = tc_desc_lo(smem_u32(tile0 + VH_A_BYTES), VH_B_LBO);
    unsigned char *laneA = tile0 + (lane >> 4) * VH_A_LBO + (lane & 15);
    unsigned char *laneB = tile0 + VH_A_BYTES + (lane >> 4) * VH_B_LBO + (lane & 15);
    uint32_t phase = 0;  // parity of this warp's barrier

    for (int r = blockIdx.x; r < A.B.n_reads; r += gridDim.x) {
        adb_record *rec = A.out + r;
        __syncthreads();
        ReadSrc gsrc;
        if (!vc_read_start(A, r, gsrc)) continue;
        VcIn I;
        if (!vc_inputs(A, cfg, r, gsrc, I)) continue;
        const int size = I.size, a_end = I.a_end;
        if (size <= 0) continue;
        if (tid == 0) H.in = I;
        // the window stays in global memory: the helpers take a 16-byte aligned base + the index of sample 0
        VfRead R;
        R.W16 = reinterpret_cast<const uint16_t *>((uintptr_t)gsrc.i16 & ~(uintptr_t)15);
        R.s0 = (int)(((uintptr_t)gsrc.i16 & 15) >> 1);
        R.n = size; R.coff = gsrc.coff; R.cscale = gsrc.cscale;
        R.kmin = 0; R.kmax = 0;
        const int16_t *W = gsrc.i16;
        if (tid == 32) {  // the next read of this CTA: its window travels to L2 while this one is worked on
            const int rn = r + gridDim.x;
            if (rn < A.B.n_reads) {
                const ReadSrc nx = make_src(A.B, rn);
                if (nx.i16 != nullptr && nx.n > 8) {
                    const uintptr_t p0 = ((uintptr_t)nx.i16 + 15) & ~(uintptr_t)15;
                    const uint32_t nbytes = (uint32_t)(((uintptr_t)(nx.i16 + nx.n) - p0) & ~(uintptr_t)15);
                    if (nbytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p0), "r"(nbytes) : "memory");
                }
            }
        }
        int cok = 1;
        const int base = gsb_code_at(VH_M == 128 ? -20.0f : 25.0f, false, R.coff, R.cscale, &cok);
        if (!cok) continue;
        vc_zero_record(rec);
#ifdef ADB_VH_STATS
        long long vh_t0 = clock64();
        if (tid == 0) atomicAdd(&vh_dbg[0], 1ull);
#endif

        // ---- speculative inputs of the checks (SURVEY A.8) ----
        int n_open = 0, op_last = 0;
        if (a_end != 0 && cfg.detect_open_pores) {
            int ok = 1;
            const int c200 = gsb_code_at(200.0f, false, R.coff, R.cscale, &ok);
            int ob = a_end;
            { int oa = 0; clip_seg(oa, ob, size); }
            if (ob + 16 > 32 * VH_OP_WORDS) continue;  // (uniform) adapter longer than the scan's bit mask: validate_kernel
            n_open = vh_open_pores(R, H, ob, c200, rec, &op_last);
        }
        const VcGeom G = vc_geometry(cfg, I, n_open, op_last);
        if (G.rr_geom) {
            float rm0, rm1;
            vf_mean_pair_t<int16_t>(W, R.coff, R.cscale, S, G.ra, G.ra + G.rlen - cfg.mean_window, cfg.mean_window, rm0, rm1);
            if (tid == 0) { S.st.rm0 = rm0; S.st.rm1 = rm1; }
        }

        VH_T(1);
        __syncthreads();
        if (warp == 0) {
            // cut points = the distinct range ends, sorted: lane l holds one end (lanes 24 / 25: 0 and size), its place is
            // the number of distinct smaller ends
            int v = (lane == 25) ? size : 0;
            bool on = lane == 24 || lane == 25;
#pragma unroll
            for (int q = 0; q < VC_NQ; q++) {
                if ((lane >> 1) == q) { v = (lane & 1) ? G.qb[q] : G.qa[q]; on = G.qb[q] > G.qa[q]; }
            }
            const unsigned onm = __ballot_sync(ADB_FULL, on);
            bool first = on;
            for (int j = 0; j < 26; j++) {
                const int vj = __shfl_sync(ADB_FULL, v, j);
                if (((onm >> j) & 1u) && j < lane && vj == v) first = false;
            }
            const unsigned fm = __ballot_sync(ADB_FULL, first);
            int pos = 0;
            for (int j = 0; j < 26; j++) {
                const int vj = __shfl_sync(ADB_FULL, v, j);
                if (((fm >> j) & 1u) && vj < v) pos++;
            }
            const int np = __popc(fm) - 1;
            if (first && pos <= VH_MAX_PIECES) H.cuts[pos] = v;
            __syncwarp();
            if (lane == 0) { H.np = np; H.n_low = 0; H.n_high = 0; H.unsettled = 0; }
        }
        if (tid < 2 * VH_MAX_PIECES) (&H.psum[0][0])[tid] = 0ull;
        // (the accumulators are all-zero: cleared by the warps that read them, right after the previous read's readout)
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int np = H.np;
        VH_T(2);
        if (np > VH_MAX_PIECES) continue;  // (uniform) more ranges than accumulators: validate_kernel
        // ---- one pass over the samples: one-hot tiles -> MMA -> clear; sums of the codes per piece on the way ----
        // A batch = 32 * VH_SUB consecutive samples of one piece (VH_SUB per lane, one MMA per 32); the batches of all
        // pieces are dealt round-robin to the warps, the samples of a warp's next batch are loaded one batch ahead.
        {
            int cmin = 0x7fffffff, cmax = -0x7fffffff;   // code range seen by this lane
            int boff = 0;                                // batches of the pieces before p
            for (int p = 0; p < np; p++) {
                const int c0 = H.cuts[p], c1 = H.cuts[p + 1];
                const int nb = (c1 - c0 + 32 * VH_SUB - 1) / (32 * VH_SUB);
                int bt = (warp - boff) & (VH_WARPS - 1);  // this warp's first batch of the piece
                boff += nb;
                if (bt >= nb) continue;
                const uint32_t dcol = tmem + (uint32_t)p * 16;
                int j = c0 + bt * (32 * VH_SUB) + lane;
                int nxt[VH_SUB];
#pragma unroll
                for (int u = 0; u < VH_SUB; u++) nxt[u] = (j + 32 * u < c1) ? (int)W[j + 32 * u] : 0;
                int s1 = 0;                              // sum of (code - base) of this lane: |code - base| < 2^16, < 2^11 batches
                unsigned long long s2 = 0;               // sum of their squares
                for (; bt < nb; bt += VH_WARPS, j += VH_WARPS * 32 * VH_SUB) {
                    int code[VH_SUB];
#pragma unroll
                    for (int u = 0; u < VH_SUB; u++) code[u] = nxt[u];
                    const int jn = j + VH_WARPS * 32 * VH_SUB;
#pragma unroll
                    for (int u = 0; u < VH_SUB; u++) nxt[u] = (jn + 32 * u < c1) ? (int)W[jn + 32 * u] : 0;
                    unsigned char *pA8[VH_SUB], *pB8[VH_SUB];
#pragma unroll
                    for (int u = 0; u < VH_SUB; u++) {
                        const bool on = j + 32 * u < c1;
                        const int dd = code[u] - base;
                        if (on) {
                            cmin = min(cmin, dd); cmax = max(cmax, dd);
                            const unsigned ud = (unsigned)abs(dd);
                            s1 += dd;
                            s2 += (unsigned long long)(ud * ud);
                        }
                        const int cp = min(max(dd, 0), VH_BINS - 1);
                        pA8[u] = laneA + u * VH_TILE_BYTES + (cp >> 4) * 16;
                        pB8[u] = laneB + u * VH_TILE_BYTES + (cp & 15) * 16;
                        if (on) { *pA8[u] = 0x38; *pB8[u] = 0x38; }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (tc_elect_one()) {
#pragma unroll
                        for (int u = 0; u < VH_SUB; u++)
                            vh_mma_f8(dcol, a_lo0 + u * (VH_TILE_BYTES >> 4), ab_hi, b_lo0 + u * (VH_TILE_BYTES >> 4), ab_hi);
                        tc_commit(&H.bar[warp]);
                    }
                    __syncwarp();
                    mbar_wait(&H.bar[warp], phase);
                    phase ^= 1;
#pragma unroll
                    for (int u = 0; u < VH_SUB; u++)
                        if (j + 32 * u < c1) { *pA8[u] = 0; *pB8[u] = 0; }
                }
                // this warp's share of the piece's sums
                long long t1 = s1;
                unsigned long long t2 = s2;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { t1 += __shfl_xor_sync(ADB_FULL, t1, o); t2 += __shfl_xor_sync(ADB_FULL, t2, o); }
                if (lane == 0) { atomicAdd(&H.psum[p][0], (unsigned long long)t1); atomicAdd(&H.psum[p][1], t2); }  // (two's complement)
            }
            const bool lo_out = __any_sync(ADB_FULL, cmin < 0), hi_out = __any_sync(ADB_FULL, cmax > VH_BINS - 1);
            if (lane == 0) { if (lo_out) atomicAdd(&H.n_low, 1); if (hi_out) atomicAdd(&H.n_high, 1); }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        VH_T(3);
        // ---- accumulators -> counts (u16) in the arena (the tiles are idle and all-zero) ----
        {
            const int quad = warp & 3;
            for (int pp = 0; pp < 4; pp++) {
                const int p = (warp >> 2) * 4 + pp;
                if (p >= np) break;
                uint32_t v[16];
                vh_tmem_ld16(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)p * 16, v);
                uint32_t w[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const unsigned c0 = (unsigned)__float2int_rn(__uint_as_float(v[2 * i]));
                    const unsigned c1 = (unsigned)__float2int_rn(__uint_as_float(v[2 * i + 1]));
                    w[i] = (c0 & 0xffffu) | (c1 << 16);
                }
                // accumulator row of this thread's TMEM lane: M = 128 -> the lane; M = 64 -> 16 rows per 32-lane quarter
                const int row = (VH_M == 128) ? quad * 32 + lane : quad * 16 + lane;
                if (VH_M == 128 || lane < 16) {
                    uint4 *dst = reinterpret_cast<uint4 *>(cum + (size_t)p * VH_BINS + row * 16);
                    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
                    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
                }
            }
            // this warp's part of the accumulators (the lanes and columns it has just read) back to zero for the next read
            const uint32_t t0 = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(warp >> 2) * 64;
            vh_tmem_zero32(t0);
            vh_tmem_zero32(t0 + 32);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- counts -> cumulative counts per piece (warp p: 8 rounds of 256 bins, 8 bins per lane) ----
        if (warp < np) {
            uint16_t *cp = cum + (size_t)warp * VH_BINS;
            unsigned carry = 0;
            for (int rd = 0; rd < VH_BINS / 256; rd++) {
                uint4 *q4 = reinterpret_cast<uint4 *>(cp + rd * 256 + lane * 8);
                const uint4 x = *q4;
                unsigned e[8] = {x.x & 0xffffu, x.x >> 16, x.y & 0xffffu, x.y >> 16, x.z & 0xffffu, x.z >> 16, x.w & 0xffffu, x.w >> 16};
#pragma unroll
                for (int i = 1; i < 8; i++) e[i] += e[i - 1];
                unsigned incl = e[7];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(ADB_FULL, incl, o); if (lane >= o) incl += t; }
                const unsigned off = carry + incl - e[7];
#pragma unroll
                for (int i = 0; i < 8; i++) e[i] += off;
                *q4 = make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
                carry += __shfl_sync(ADB_FULL, incl, 31);
            }
        }
        __syncthreads();
        VH_T(4);
        // ---- the statistics: rank query q on warp q % 8 (32-way searches), then the four MADs on warps 0..3 ----
        {
            const int n_low = H.n_low, n_high = H.n_high;
            for (int qq = warp; qq < VC_NQ; qq += VH_WARPS) {
                int a = 0, b = 0;
#pragma unroll
                for (int q = 0; q < VC_NQ; q++) if (qq == q) { a = G.qa[q]; b = G.qb[q]; }
                int v0 = 0, v1 = 0;
                const int n = b - a;
                if (n > 0) {
                    const VhRange q = vh_range(H, a, b, size);
                    bool two;
                    const int k = vc_rank(qq, n, two);
                    const int x0 = vh_wselect(cum, q.p0, q.p1, k);
                    const int x1 = two ? vh_wselect(cum, q.p0, q.p1, k + 1) : x0;
                    if (((x0 <= 0 || x1 <= 0) && n_low > 0) || ((x0 >= VH_BINS - 1 || x1 >= VH_BINS - 1) && n_high > 0)) H.unsettled = 1;
                    v0 = x0 + base;
                    v1 = x1 + base;
                }
                if (lane == 0) { S.st.c0[qq] = v0; S.st.c1[qq] = v1; S.st.n[qq] = n; }
            }
        }
        __syncthreads();
        // the four MADs (ranges 0, 1, 4, 9): warp w searches the right side of range w & 3 (w < 4) or its left side
        {
            const int t = warp & 3;
            const int src = (t == 0) ? VC_A0 : (t == 1) ? VC_A1 : (t == 2) ? VC_P : VC_R;
            int a = 0, b = 0;
#pragma unroll
            for (int q = 0; q < VC_NQ; q++) if (src == q) { a = G.qa[q]; b = G.qb[q]; }
            const int n = b - a;
            const float med = vc_median(S.st, src, R.coff, R.cscale);
            const bool live = n > 0 && med == med;
            const VhMad M(R, H, cum, vh_range(H, a, b, size), base, max(n, 1), live ? med : 0.0f);
            if (live) { const int f = M.first_pass(warp < 4); if (lane == 0) H.mfp[t][warp >> 2] = f; }
            __syncthreads();
            if (warp < 4) {
                const float mad = live ? M.finish(H.mfp[t][0], H.mfp[t][1]) : CUDART_NAN_F;
                if (lane == 0) S.st.mad[t] = mad;
            }
        }
        __syncthreads();
        const bool unsettled = H.unsettled != 0;
        VH_T(5);
        __syncthreads();
        // the part of the arena that held the cumulative counts goes back to all-zero operand tiles for the next read
        for (int i = tid; i < np * (VH_BINS * 2 / 16); i += VF_THREADS) reinterpret_cast<uint4 *>(arena)[i] = make_uint4(0, 0, 0, 0);
        VH_T(6);
        if (unsettled) continue;  // (uniform) codes outside the histogram range matter: validate_kernel

        // ---- the checks (adb_vcheck.cuh) on warp 0 only ----
        // (scalar work, much of it float64: run redundantly on all eight warps it takes issue slots and instruction
        // fetch from the other CTAs of the SM -- measured 14.0 -> 13.3 ms per 100k RNA002 reads; the other warps wait at
        // the top of the loop)
        if (warp == 0) {
            if (lane == 0) vc_small_mean_var(H.in, W, S.st);
            __syncwarp();
            const VcOut o = vc_checks(cfg, H.in, G, S.st, A.mode, A.cand_followup != 0);
            if (!o.defer) {  // (else validate_kernel redoes this read from scratch)
                // partition mean / std (S.dtmp[0..2] / [3..5]) from the exact per-piece sums of the pass above (three
                // lanes, one partition each)
                __syncwarp();
                if (lane < 3) {
                    int a, b;
                    double pm = CUDART_NAN, ps = CUDART_NAN;
                    vc_partition(H.in, o, lane, a, b);
                    clip_seg(a, b, size);
                    const int n = b - a;
                    if (n > 0) {
                        const VhRange q = vh_range(H, a, b, size);
                        long long d1 = 0, d2 = 0;
                        for (int p = q.p0; p < q.p1; p++) { d1 += (long long)H.psum[p][0]; d2 += (long long)H.psum[p][1]; }
                        const long long s1 = d1 + (long long)n * base;                                   // sum of the codes
                        const long long s2 = d2 + 2ll * base * d1 + (long long)n * base * (long long)base;  // sum of their squares
                        vc_mean_std(s1, s2, n, R.coff, R.cscale, pm, ps);
                    }
                    S.dtmp[lane] = pm; S.dtmp[3 + lane] = ps;
                }
                __syncwarp();
                if (!(o.valid & ADB_V_OPEN_PORES) || o.exception) {
                    for (int i = lane; i < ADB_MAX_OPEN_PORES; i += 32) rec->open_pores[i] = 0;  // the scan was speculative
                }
                if (tid == 0) {
                    vc_write_spec_record(rec, H.in, S.st, o, S.dtmp, S.dtmp + 3);
                    A.done[r] = o.followup ? 2 : 1;  // (read by the kernels launched behind this one: no fence needed)
                }
            }
        }
        VH_T(7);
    }
    __syncthreads();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem));
}
