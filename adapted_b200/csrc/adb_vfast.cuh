// validate_boundaries + per-segment statistics for int16 sources WITHOUT shared-memory atomics.
//
// Reference: adapted/detect/combined.py:358-631 (the checks and the record: adb_vcheck.cuh, SURVEY.md A.8).
//
// The histogram-based statistics of adb_validate.cuh are bound by the shared-memory atomic unit (~2 cycles per
// sample and histogram, ncu: profiles/r1_validate_kernel_v3.txt).  Here every order statistic of a read is found by
// COUNTING: the staged window of non-negative int16 ADC codes is read as packed half-precision bit patterns (for
// 0 <= code < 0x7c00 the integer order and the fp16 order coincide), one HSET2.LE compares two samples with a probe
// and the 0xffff / 0 lane masks are summed with plain integer adds.  All statistics of a read advance together:
//   round A  bisection on the code value for every rank needed (medians, p15 / p85 of numpy's linear percentile),
//   round B  bisection for the k-th smallest |pA(code) - med| (MAD): deviations are monotone on either side of the
//            median, so "how many samples deviate at most t" is the count of one code interval whose ends are found
//            by evaluating the float32 deviations exactly; the candidates of both sides are halved together by
//            probing the middle candidate of the longer side.
// Sums for mean / std are exact integer sums of the codes.  The float32 moving-statistics series (bottleneck
// recurrences, mvs_series_kernel) are staged in shared memory and their medians found by bisection on the ordered
// float bits.  The checks and the record are those of adb_vcheck.cuh.  Further poly(A) candidates after a failed first
// one go to validate_cand_kernel (below); anything else outside this path (float32 sources, codes outside [0, 0x7c00),
// no precomputed series, the CNN path's hail-mary fallback) is left to validate_kernel, which skips the reads flagged
// done here.
#pragma once
#include <cuda_fp16.h>

#include "adb_common.cuh"
#include "adb_gsample.cuh"
#include "adb_validate.cuh"
#include "adb_series_median.cuh"
#include "adb_vcheck.cuh"

#define VF_THREADS 256
#define VF_MAX_TASKS 12
#define VF_KEY_LIMIT 0x7c00

struct VfTask {
    int a, b;      // sample range [a, b) of the window
    int kind;      // 0: rank (count of codes <= idx); 1: k-th smallest deviation from the median (MAD)
    int k;         // 0-based rank looked for
    int lo, hi;    // search interval over the index; hi = first index whose count exceeds k (or the sentinel)
    int cnt_hi;    // count at hi
    int pv;        // deviation search: first code whose value is >= med
    float med;
    int sent;      // sentinel: hi == sent means "no index of this task satisfies the predicate"
    int smin, smax;  // code bounds of the samples of the segment
    // deviation search: candidates still undecided on the right side (codes pv + i, i in [rlo, rhi)) and on the left
    // side (codes pv - 1 - i, i in [llo, lhi)); candidates below the lows fail the predicate, from the his on they pass
    int rlo, rhi, llo, lhi;
    int jL, jR;    // codes pv - jL .. pv + jR - 1 deviate at most t_probe
    float t_probe; // deviation probed in the running pass
    float t_best;  // smallest deviation found so far that passes, and the count of samples deviating at most that much
    int c_best;
    int pA, pB;    // probes of the running pass: count the codes in [pA, pB]
    int mid;
    int active;
    // scan geometry, fixed per task: full 16-byte vectors [v0, v1) of W16, `voff` = offset of v0 in the flattened
    // vector space of all tasks of the round, boundary elements [hb, he) and [tb, te) (W16 indices, < 8 each)
    int v0, v1, voff;
    int hb, he, tb, te;
};

struct VfScratch {  // shared memory
    VfTask task[VF_MAX_TASKS];
    unsigned cnt[VF_MAX_TASKS];
    int ntask;
    int vtotal;    // vectors of all tasks of the round
    ushort4 items[VF_THREADS / 32][VF_MAX_TASKS];  // per warp: (task, first vector, end vector, owns the boundary elements)
    int nitems[VF_THREADS / 32];
    unsigned tmin[VF_MAX_TASKS], tmax[VF_MAX_TASKS];  // per-task code bounds (vf_task_bounds)
    uint32_t cand[2][64];  // keys left inside the brackets of vf_series_medians
    int ncand[2];
    int itmp[16];
    unsigned wtot[8];
    long long ltmp[8];
    float ftmp[8];
    double dtmp[8];
    uint32_t utmp[8];
    VcStats st;    // what the counting passes hand over to the checks (adb_vcheck.cuh)
    VcOut out;     // their outcome (validate_fast_kernel: thread 0 runs the checks)
};

struct VfRead {      // per-read constants (registers)
    const uint16_t *W16;  // 16-byte aligned base of the staged window
    int s0;               // index of sample 0 in W16
    int n;                // samples in the window
    float coff, cscale;
    int kmin, kmax;       // code bounds of the window
};

__device__ __forceinline__ float vf_pa(const VfRead &R, int code) { return gsb_pa(code, R.coff, R.cscale); }

__device__ __forceinline__ unsigned vf_decode(unsigned s) {
    // s = sum of HSET2 lane masks (0xffff per true half): recover the number of true halves
    const unsigned nlo = (0u - s) & 0xffffu;
    const unsigned t = ((s + nlo) >> 16) & 0xffffu;
    const unsigned nhi = (nlo - t) & 0xffffu;
    return nlo + nhi;
}

__device__ __forceinline__ __half2 vf_h2(unsigned code) {
    const unsigned w = (code & 0xffffu) * 0x00010001u;
    return *reinterpret_cast<const __half2 *>(&w);
}

// scan geometry of the window range [a, b) (a < b)
__device__ __forceinline__ void vf_geometry(const VfRead &R, VfTask &t, int a, int b, int voff) {
    const int i0 = R.s0 + a, i1 = R.s0 + b;
    const int v0 = (i0 + 7) >> 3, v1 = max(i1 >> 3, v0);
    t.v0 = v0; t.v1 = v1; t.voff = voff;
    t.hb = i0; t.he = min(i1, v0 << 3);
    t.tb = max(v1 << 3, t.he); t.te = i1;
}

// per-lane partial of: number of samples in the full vectors [vb, ve) of W16 whose code lies in [pA, pB] (pA <= pB).
// Two vectors per iteration, both loads issued before the compares.
__device__ __forceinline__ int vf_count_vectors(const VfRead &R, int vb, int ve, int pA, int pB) {
    const int lane = threadIdx.x & 31;
    const uint4 *V = reinterpret_cast<const uint4 *>(R.W16);
    const __half2 hB = vf_h2((unsigned)pB);
    unsigned sB = 0, sA = 0;
    if (pA > 0) {
        const __half2 hA = vf_h2((unsigned)(pA - 1));
        auto eat = [&](const uint4 &q) {
            const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const __half2 h = *reinterpret_cast<const __half2 *>(&w[t]);
                sB += __hle2_mask(h, hB);
                sA += __hle2_mask(h, hA);
            }
        };
        int v = vb + lane;
        for (; v + 32 < ve; v += 64) {
            const uint4 qa = V[v], qb = V[v + 32];
            eat(qa);
            eat(qb);
        }
        if (v < ve) eat(V[v]);
        return (int)vf_decode(sB) - (int)vf_decode(sA);
    }
    auto eat1 = [&](const uint4 &q) {
        const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int t = 0; t < 4; t++) sB += __hle2_mask(*reinterpret_cast<const __half2 *>(&w[t]), hB);
    };
    int v = vb + lane;
    for (; v + 32 < ve; v += 64) {
        const uint4 qa = V[v], qb = V[v + 32];
        eat1(qa);
        eat1(qb);
    }
    if (v < ve) eat1(V[v]);
    return (int)vf_decode(sB);
}

// float32 deviation of a code from the median, as the reference computes it on the pA values
__device__ __forceinline__ float vf_dev(const VfRead &R, int code, float med) { return fabsf(__fsub_rn(vf_pa(R, code), med)); }

// deviation of the i-th candidate of a side (right: code pv + i, left: code pv - 1 - i); non-decreasing in i
__device__ __forceinline__ float vf_side_dev(const VfRead &R, const VfTask &t, bool right, int i) {
    return vf_dev(R, right ? t.pv + i : t.pv - 1 - i, t.med);
}

// first index of a side (n candidates) whose deviation is > t (strict) or >= t: the calibration is nearly linear, so
// t / scale is within a step or two of the answer; the guess is corrected by exact float32 evaluations
__device__ int vf_side_first(const VfRead &R, const VfTask &t, bool right, int n, float thr, bool strict) {
    float gf = thr / R.cscale;
    int g = (gf == gf && gf < 1e9f) ? (int)gf : n;
    g = min(max(g, 0), n);
    int guard = 0;
    while (g > 0 && guard++ < 100000) {
        const float d = vf_side_dev(R, t, right, g - 1);
        if (strict ? (d > thr) : (d >= thr)) g--; else break;
    }
    while (g < n && guard++ < 100000) {
        const float d = vf_side_dev(R, t, right, g);
        if (strict ? !(d > thr) : !(d >= thr)) g++; else break;
    }
    return g;
}

__device__ __forceinline__ bool vf_pending(const VfTask &t) {
    return t.kind == 0 ? (t.lo < t.hi) : (t.rlo < t.rhi || t.llo < t.lhi);
}

// choose the probe of the next pass (one thread); false when the task has converged
__device__ bool vf_prepare(const VfRead &R, VfTask &t) {
    if (!vf_pending(t)) { t.active = 0; return false; }
    t.active = 1;
    if (t.kind == 0) { t.mid = (t.lo + t.hi) >> 1; t.pA = 0; t.pB = t.mid; return true; }
    // the middle candidate of the longer side: by symmetry of the two sides it halves the other one as well
    const int nR = t.smax + 1 - t.pv, nL = t.pv - t.smin;
    const bool right = (t.rhi - t.rlo) >= (t.lhi - t.llo);
    const int i = right ? (t.rlo + t.rhi) >> 1 : (t.llo + t.lhi) >> 1;
    const float thr = vf_side_dev(R, t, right, i);
    t.t_probe = thr;
    t.jR = vf_side_first(R, t, true, nR, thr, true);
    t.jL = vf_side_first(R, t, false, nL, thr, true);
    t.pA = t.pv - t.jL;
    t.pB = t.pv + t.jR - 1;
    return true;
}

// take the count of the pass (one thread)
__device__ void vf_update(const VfRead &R, VfTask &t, int c) {
    if (t.kind == 0) {
        if (c > t.k) { t.hi = t.mid; t.cnt_hi = c; } else t.lo = t.mid + 1;
        return;
    }
    if (c > t.k) {
        // every candidate deviating at least t_probe passes
        const int nR = t.smax + 1 - t.pv, nL = t.pv - t.smin;
        t.rhi = min(t.rhi, vf_side_first(R, t, true, nR, t.t_probe, false));
        t.lhi = min(t.lhi, vf_side_first(R, t, false, nL, t.t_probe, false));
        t.rlo = min(t.rlo, t.rhi);
        t.llo = min(t.llo, t.lhi);
        t.t_best = t.t_probe;
        t.c_best = c;
    } else {
        // every candidate deviating at most t_probe fails
        t.rlo = min(max(t.rlo, t.jR), t.rhi);
        t.llo = min(max(t.llo, t.jL), t.lhi);
    }
}

__device__ void vf_build_items(VfScratch &S, bool all_tasks) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ntask = S.ntask;
    const int nw = VF_THREADS / 32;
    if (lane == 0) {
        const int wbeg = (int)(((long long)S.vtotal * warp) / nw), wend = (int)(((long long)S.vtotal * (warp + 1)) / nw);
        int n = 0;
        for (int q = 0; q < ntask; q++) {
            const VfTask &t = S.task[q];
            if (!all_tasks && !vf_pending(t)) continue;
            const int fb = max(t.voff, wbeg), fe = min(t.voff + (t.v1 - t.v0), wend);
            const int edge = (warp == (q & (nw - 1))) && (t.hb < t.he || t.tb < t.te);
            if (fb < fe) S.items[warp][n++] = make_ushort4((unsigned short)q, (unsigned short)(t.v0 + (fb - t.voff)), (unsigned short)(t.v0 + (fe - t.voff)), (unsigned short)edge);
            else if (edge) S.items[warp][n++] = make_ushort4((unsigned short)q, 0, 0, 1);
        }
        S.nitems[warp] = n;
    }
    __syncwarp();
}

// code bounds of the samples of every (rank) task: the bisections then start from the segment's own range instead of
// the window's (an open-pore stretch or a spike elsewhere in the read would cost every task three more passes).
// CTA-wide; sets lo / hi / smin / smax of every task.
__device__ void vf_task_bounds(const VfRead &R, VfScratch &S) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __syncthreads();
    const int ntask = S.ntask;
    if (tid < ntask) { S.tmin[tid] = 0xffffu; S.tmax[tid] = 0u; }
    vf_build_items(S, true);
    __syncthreads();
    const uint4 *V = reinterpret_cast<const uint4 *>(R.W16);
    const int nit = S.nitems[warp];
    for (int it = 0; it < nit; it++) {
        const ushort4 item = S.items[warp][it];
        const VfTask &t = S.task[item.x];
        unsigned mn = 0xffffffffu, mx = 0u;
        for (int v = item.y + lane; v < item.z; v += 32) {
            const uint4 q = V[v];
            mn = __vminu2(__vminu2(mn, q.x), __vminu2(q.y, __vminu2(q.z, q.w)));
            mx = __vmaxu2(__vmaxu2(mx, q.x), __vmaxu2(q.y, __vmaxu2(q.z, q.w)));
        }
        unsigned lo = min(mn & 0xffffu, mn >> 16), hi = max(mx & 0xffffu, mx >> 16);
        if (item.w && lane < 16) {
            const int i = (lane < 8) ? t.hb + lane : t.tb + (lane - 8);
            const int iend = (lane < 8) ? t.he : t.te;
            if (i < iend) { const unsigned code = R.W16[i]; lo = min(lo, code); hi = max(hi, code); }
        }
        lo = __reduce_min_sync(ADB_FULL, lo);
        hi = __reduce_max_sync(ADB_FULL, hi);
        if (lane == 0) { atomicMin(&S.tmin[item.x], lo); atomicMax(&S.tmax[item.x], hi); }
    }
    __syncthreads();
    if (tid < ntask) {
        VfTask &t = S.task[tid];
        t.smin = (int)S.tmin[tid]; t.smax = (int)S.tmax[tid];
        t.lo = t.smin; t.hi = t.smax; t.sent = t.smax + 1;
    }
}

__device__ void vf_run(const VfRead &R, VfScratch &S) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __syncthreads();
    const int ntask = S.ntask;
    vf_build_items(S, false);
    bool mine = false;
    if (tid < ntask) {
        VfTask &t = S.task[tid];
        S.cnt[tid] = 0;
        mine = vf_prepare(R, t);
    }
    const int nit = S.nitems[warp];
    while (__syncthreads_or(mine)) {
        for (int it = 0; it < nit; it++) {
            const ushort4 item = S.items[warp][it];
            const VfTask &t = S.task[item.x];
            if (!t.active) continue;
            const int pA = t.pA, pB = t.pB;
            if (pB < pA) continue;
            int c = 0;
            if (item.y < item.z) c = vf_count_vectors(R, item.y, item.z, pA, pB);
            if (item.w && lane < 16) {
                const int i = (lane < 8) ? t.hb + lane : t.tb + (lane - 8);
                const int iend = (lane < 8) ? t.he : t.te;
                if (i < iend) { const int code = R.W16[i]; c += (code >= pA && code <= pB); }
            }
            c = __reduce_add_sync(ADB_FULL, c);
            if (lane == 0 && c) atomicAdd(&S.cnt[item.x], (unsigned)c);
        }
        __syncthreads();
        mine = false;
        if (tid < ntask) {
            VfTask &t = S.task[tid];
            if (t.active) {
                const int c = (int)S.cnt[tid];
                S.cnt[tid] = 0;
                vf_update(R, t, c);
                mine = vf_prepare(R, t);
            }
        }
    }
}

// smallest code > v (succ) / largest code < v (pred) among the samples [a, b); CTA-wide, rare path.  -1 if none.
__device__ int vf_neighbour(const VfRead &R, VfScratch &S, int a, int b, int v, bool succ) {
    __syncthreads();
    if (threadIdx.x == 0) S.itmp[15] = succ ? 0x7fffffff : -1;
    __syncthreads();
    int best = succ ? 0x7fffffff : -1;
    for (int j = a + threadIdx.x; j < b; j += blockDim.x) {
        const int c = R.W16[R.s0 + j];
        if (succ) { if (c > v) best = min(best, c); } else { if (c < v) best = max(best, c); }
    }
    if (succ) { if (best != 0x7fffffff) atomicMin(&S.itmp[15], best); } else { if (best >= 0) atomicMax(&S.itmp[15], best); }
    __syncthreads();
    const int r = S.itmp[15];
    __syncthreads();
    return (r == 0x7fffffff) ? -1 : r;
}

// ---- staging helpers ---------------------------------------------------------------------------------------------
// min / max code of the window (packed int16 min / max, VIMNMX.S16x2).  CTA-wide.
__device__ void vf_minmax(const VfRead &R, VfScratch &S, int &kmin, int &kmax) {
    const int tid = threadIdx.x;
    const int i0 = R.s0, i1 = R.s0 + R.n;
    const int v0 = (i0 + 7) >> 3, v1 = i1 >> 3;
    const int head_end = min(i1, v0 << 3), tail_beg = max(v1 << 3, head_end);
    int lo = 0x7fff, hi = -0x8000;
    if (tid < 8) { const int i = i0 + tid; if (i < head_end) { const int c = (int16_t)R.W16[i]; lo = min(lo, c); hi = max(hi, c); } }
    else if (tid < 16) { const int i = tail_beg + tid - 8; if (i < i1) { const int c = (int16_t)R.W16[i]; lo = min(lo, c); hi = max(hi, c); } }
    unsigned mn = 0x7fff7fffu, mx = 0x80008000u;
    const uint4 *V = reinterpret_cast<const uint4 *>(R.W16);
    for (int v = v0 + tid; v < v1; v += VF_THREADS) {
        const uint4 q = V[v];
        mn = __vmins2(__vmins2(mn, q.x), __vmins2(q.y, __vmins2(q.z, q.w)));
        mx = __vmaxs2(__vmaxs2(mx, q.x), __vmaxs2(q.y, __vmaxs2(q.z, q.w)));
    }
    lo = min(lo, min((int)(int16_t)(mn & 0xffffu), (int)(int16_t)(mn >> 16)));
    hi = max(hi, max((int)(int16_t)(mx & 0xffffu), (int)(int16_t)(mx >> 16)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(ADB_FULL, lo, o));
        hi = max(hi, __shfl_xor_sync(ADB_FULL, hi, o));
    }
    __syncthreads();
    if ((tid & 31) == 0) { S.itmp[tid >> 5] = lo; S.itmp[8 + (tid >> 5)] = hi; }
    __syncthreads();
    lo = 0x7fff; hi = -0x8000;
    for (int w = 0; w < VF_THREADS / 32; w++) { lo = min(lo, S.itmp[w]); hi = max(hi, S.itmp[8 + w]); }
    __syncthreads();
    kmin = lo; kmax = hi;
}

// find_open_pores (anomalies.py:15-35) on codes: a sample is an open-pore sample iff code >= c200.  Same structure
// as open_pores_scan in adb_validate.cuh.
__device__ int vf_open_pores(const VfRead &R, VfScratch &S, int a, int b, int c200, adb_record *rec, int *last) {
    clip_seg(a, b, R.n);
    const int n = b - a;
    const int T = blockDim.x, tid = threadIdx.x;
    const int chunk = (n + T - 1) / T;
    const int j0 = min(tid * chunk, n), j1 = min(j0 + chunk, n);
    const uint16_t *w = R.W16 + R.s0 + a;
    int *sh = S.itmp;  // [0]=hits [1]=first hit [2]=last hit [4]=last valid
    __syncthreads();
    if (tid == 0) { sh[0] = 0; sh[1] = 0x7fffffff; sh[2] = -1; sh[3] = 0; sh[4] = -1; }
    __syncthreads();
    int hits = 0, first = 0x7fffffff, lastp = -1, ncand = 0, lastc = -1;
    for (int j = j0; j < j1; j++) {
        if ((int)w[j] >= c200) {
            hits++;
            first = min(first, j);
            lastp = j;
            bool gap = true;
            for (int k = 1; k < 10 && gap; k++)
                if (j - k >= 0 && (int)w[j - k] >= c200) gap = false;
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
        if (first_hit >= j0 && first_hit < j1) { ncand--; if (lastc == first_hit) lastc = -1; }
        int incl = ncand;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(ADB_FULL, incl, o);
            if ((tid & 31) >= o) incl += v;
        }
        __syncthreads();
        if ((tid & 31) == 31) S.wtot[tid >> 5] = (unsigned)incl;
        if (lastc >= 0) atomicMax(&sh[4], lastc);
        __syncthreads();
        int wbase = 0, total = 0;
        for (int q = 0; q < (int)((T + 31) >> 5); q++) {
            if (q < (tid >> 5)) wbase += (int)S.wtot[q];
            total += (int)S.wtot[q];
        }
        int pos = wbase + incl - ncand;
        if (total > 0) {
            if (ncand > 0 && pos < ADB_MAX_OPEN_PORES) {
                for (int j = j0; j < j1 && pos < ADB_MAX_OPEN_PORES; j++) {
                    if (j == first_hit) continue;
                    if ((int)w[j] >= c200) {
                        bool gap = true;
                        for (int k = 1; k < 10 && gap; k++)
                            if (j - k >= 0 && (int)w[j - k] >= c200) gap = false;
                        if (gap) rec->open_pores[pos++] = a + j;
                    }
                }
            }
            result_n = total;
            *last = a + sh[4];
        } else {
            result_n = 1;
            if (tid == 0) rec->open_pores[0] = a + last_hit;
            *last = a + last_hit;
        }
    }
    __syncthreads();
    return result_n;
}

// numpy float32 mean of the `n` samples starting at a0 and at a1 (real_range_check: first / last mean_window samples)
// in numpy's pairwise order.  For 128 < n <= 512 the (at most four) leaves of the pairwise tree are summed by
// different threads and combined in tree order; other sizes by one thread per mean.  CTA-wide.
template <class T>  // uint16_t: non-negative codes of the staged window; int16_t: any code (adb_vhist.cuh)
__device__ void vf_mean_pair_t(const T *w, float coff, float cscale, VfScratch &S, int a0, int a1, int n, float &m0, float &m1) {
    __syncthreads();
    const int tid = threadIdx.x;
    if (n > 128 && n <= 512) {
        // tree: n -> (h0, n - h0); each part p > 128 -> (p2, p - p2)
        if (tid < 8) {
            const int which = tid >> 2, leaf = tid & 3;
            const int base = which ? a1 : a0;
            int h0 = n / 2; h0 -= h0 % 8;
            const int part = leaf >> 1;              // 0: left half, 1: right half
            const int pbase = part ? h0 : 0, plen = part ? n - h0 : h0;
            int lbase, llen;
            if (plen > 128) {
                int p2 = plen / 2; p2 -= p2 % 8;
                lbase = pbase + ((leaf & 1) ? p2 : 0);
                llen = (leaf & 1) ? plen - p2 : p2;
            } else {
                lbase = pbase;
                llen = (leaf & 1) ? 0 : plen;       // single leaf: the odd slot is unused
            }
            float sum = 0.f;
            if (llen > 0) {
                const T *p = w + base + lbase;
                sum = np_sum_f32_leaf([&](int i) { return __fmul_rn(__fadd_rn((float)(int)p[i], coff), cscale); }, llen);
            }
            S.ftmp[tid] = sum;
        }
        __syncthreads();
        auto combine = [&](int which) {
            int h0 = n / 2; h0 -= h0 % 8;
            const float *f = S.ftmp + which * 4;
            const float left = (h0 > 128) ? __fadd_rn(f[0], f[1]) : f[0];
            const float right = (n - h0 > 128) ? __fadd_rn(f[2], f[3]) : f[2];
            return __fdiv_rn(__fadd_rn(left, right), (float)n);
        };
        m0 = combine(0);
        m1 = combine(1);
    } else {
        if (tid == 0 || tid == 32) {
            const T *p = w + (tid == 0 ? a0 : a1);
            const float s = np_sum_f32([&](int i) { return __fmul_rn(__fadd_rn((float)(int)p[i], coff), cscale); }, n);
            S.ftmp[tid == 0 ? 0 : 1] = __fdiv_rn(s, (float)n);
        }
        __syncthreads();
        m0 = S.ftmp[0];
        m1 = S.ftmp[1];
    }
    __syncthreads();
}

__device__ __forceinline__ void vf_mean_pair(const VfRead &R, VfScratch &S, int a0, int a1, int n, float &m0, float &m1) {
    vf_mean_pair_t<uint16_t>(R.W16 + R.s0, R.coff, R.cscale, S, a0, a1, n, m0, m1);
}

// exact integer sums of the codes of up to three segments [sa[i], sb[i]) (clipped; skipped unless on[i]) -> mean /
// population std of the pA values (vc_mean_std).  CTA-wide.
__device__ void vf_mean_std3(const VfRead &R, VfScratch &S, const int sa[3], const int sb[3], const bool on[3],
                             double mean_out[3], double std_out[3]) {
    const int tid = threadIdx.x;
    __syncthreads();
    if (tid < 6) S.ltmp[tid] = 0;
    __syncthreads();
    const uint16_t *w = R.W16 + R.s0;
    int na[3];
    for (int sgm = 0; sgm < 3; sgm++) {
        int a = sa[sgm], b = sb[sgm];
        clip_seg(a, b, R.n);
        na[sgm] = on[sgm] ? b - a : 0;
        if (na[sgm] <= 0) continue;
        // 16-byte vectors over the aligned body, the (< 8 each) head / tail elements by the first threads; codes are
        // non-negative and below 0x7c00: a thread's sum of codes fits 32 bits, the squares accumulate in 64
        unsigned s1u = 0;
        unsigned long long s2u = 0;
        {
            const int i0 = R.s0 + a, i1 = R.s0 + b;
            const int v0 = (i0 + 7) >> 3, v1 = max(i1 >> 3, v0);
            const int he = min(i1, v0 << 3), tb = max(v1 << 3, he);
            const uint4 *V = reinterpret_cast<const uint4 *>(R.W16);
            for (int v = v0 + tid; v < v1; v += VF_THREADS) {
                const uint4 q = V[v];
                const unsigned ww[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    const unsigned lo = ww[t] & 0xffffu, hi = ww[t] >> 16;
                    s1u += lo + hi;
                    s2u += (unsigned long long)lo * lo;
                    s2u += (unsigned long long)hi * hi;
                }
            }
            if (tid < 16) {
                const int i = (tid < 8) ? i0 + tid : tb + (tid - 8);
                const int iend = (tid < 8) ? he : i1;
                if (i < iend) { const unsigned c = R.W16[i]; s1u += c; s2u += (unsigned long long)c * c; }
            }
        }
        long long s1 = (long long)s1u, s2 = (long long)s2u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(ADB_FULL, s1, o); s2 += __shfl_xor_sync(ADB_FULL, s2, o); }
        if ((tid & 31) == 0) {
            atomicAdd((unsigned long long *)&S.ltmp[2 * sgm], (unsigned long long)s1);
            atomicAdd((unsigned long long *)&S.ltmp[2 * sgm + 1], (unsigned long long)s2);
        }
    }
    __syncthreads();
    for (int sgm = 0; sgm < 3; sgm++) {
        const int n = na[sgm];
        if (n <= 0) { mean_out[sgm] = CUDART_NAN; std_out[sgm] = CUDART_NAN; continue; }
        vc_mean_std(S.ltmp[2 * sgm], S.ltmp[2 * sgm + 1], n, R.coff, R.cscale, mean_out[sgm], std_out[sgm]);
    }
    __syncthreads();
}

// np.nanmedian of up to two NaN-free float32 series (global memory) staged as ordered keys in `buf` (shared memory):
// bisection on the key value, both series advancing in the same passes, until at most VF_NCAND keys are left inside
// the bracket; those are gathered and ranked directly (float keys are nearly all distinct, so isolating a single key
// by bisection would take ~22 passes; isolating 64 of ~3000 takes ~6).  CTA-wide.
#define VF_NCAND 64
// STAGED = false (series longer than `buf`: poly(A) segments beyond half the window, the long-poly(A) stress set): every
// pass reads the 16-byte aligned rows from the pools (L2 resident) and forms the keys on the fly -- same passes, same
// result.
template <bool STAGED>
__device__ void vf_series_medians(VfScratch &S, const float *g0, int n0, const float *g1, int n1, uint32_t *buf, float out[2]) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *k0 = buf, *k1 = buf + ((n0 + 3) & ~3);
    __syncthreads();
    uint32_t mn[2] = {0xffffffffu, 0xffffffffu}, mx[2] = {0u, 0u};
    for (int j = tid; j < n0; j += VF_THREADS) { const uint32_t k = f32_key(g0[j]); if (STAGED) k0[j] = k; mn[0] = min(mn[0], k); mx[0] = max(mx[0], k); }
    for (int j = tid; j < n1; j += VF_THREADS) { const uint32_t k = f32_key(g1[j]); if (STAGED) k1[j] = k; mn[1] = min(mn[1], k); mx[1] = max(mx[1], k); }
    for (int q = 0; q < 2; q++) { mn[q] = warp_min_u(mn[q]); mx[q] = warp_max_u(mx[q]); }
    if (tid < 4) S.utmp[tid] = (tid < 2) ? 0xffffffffu : 0u;
    if (tid < 6) S.cnt[tid] = 0;
    if (tid < 2) S.ncand[tid] = 0;
    __syncthreads();
    if (lane == 0) {
        atomicMin(&S.utmp[0], mn[0]); atomicMin(&S.utmp[1], mn[1]);
        atomicMax(&S.utmp[2], mx[0]); atomicMax(&S.utmp[3], mx[1]);
    }
    __syncthreads();
    // search state in registers (identical in every thread): keys in [lo, hi] hold the ranks cnt_lo .. cnt_hi - 1
    uint32_t lo[2] = {S.utmp[0], S.utmp[1]}, hi[2] = {S.utmp[2], S.utmp[3]};
    const int nn[2] = {n0, n1};
    const uint32_t *kk[2] = {k0, k1};
    const float *gg[2] = {g0, g1};
    auto key_at = [&](int q, int j) -> uint32_t { return STAGED ? kk[q][j] : f32_key(gg[q][j]); };
    const unsigned rank[2] = {n0 > 0 ? (unsigned)(n0 - 1) / 2 : 0u, n1 > 0 ? (unsigned)(n1 - 1) / 2 : 0u};
    unsigned cnt_hi[2] = {(unsigned)n0, (unsigned)n1}, cnt_lo[2] = {0u, 0u};
    auto open = [&](int q) { return nn[q] > 0 && lo[q] < hi[q] && cnt_hi[q] - cnt_lo[q] > VF_NCAND; };
    int pass = 0;
    while (open(0) || open(1)) {
        uint32_t mid[2];
        for (int q = 0; q < 2; q++) {
            mid[q] = lo[q] + ((hi[q] - lo[q]) >> 1);
            if (!open(q)) continue;
            int c = 0;
            const int nv = nn[q] >> 2;
            if (STAGED) {
                const uint4 *V = reinterpret_cast<const uint4 *>(kk[q]);
                for (int v = tid; v < nv; v += VF_THREADS) {
                    const uint4 x = V[v];
                    c += (x.x <= mid[q]) + (x.y <= mid[q]) + (x.z <= mid[q]) + (x.w <= mid[q]);
                }
            } else {
                const float4 *V = reinterpret_cast<const float4 *>(gg[q]);
                for (int v = tid; v < nv; v += VF_THREADS) {
                    const float4 x = V[v];
                    c += (f32_key(x.x) <= mid[q]) + (f32_key(x.y) <= mid[q]) + (f32_key(x.z) <= mid[q]) + (f32_key(x.w) <= mid[q]);
                }
            }
            const int j = (nv << 2) + tid;
            if (j < nn[q]) c += (key_at(q, j) <= mid[q]);
            c = __reduce_add_sync(ADB_FULL, c);
            if (lane == 0 && c) atomicAdd(&S.cnt[q + 2 * (pass % 3)], (unsigned)c);
        }
        __syncthreads();
        for (int q = 0; q < 2; q++) {
            if (!open(q)) continue;
            const unsigned c = S.cnt[q + 2 * (pass % 3)];
            if (c > rank[q]) { hi[q] = mid[q]; cnt_hi[q] = c; } else { lo[q] = mid[q] + 1; cnt_lo[q] = c; }
        }
        // three rotating counter sets: the set of the previous pass has been read by everybody (this pass's barrier
        // lies in between) and is not used again before the pass after next
        if (tid < 2) S.cnt[tid + 2 * ((pass + 2) % 3)] = 0;
        pass++;
    }
    // gather the keys left in the brackets (cnt_hi - cnt_lo of them, or all equal keys when lo == hi)
    for (int q = 0; q < 2; q++) {
        if (nn[q] <= 0 || lo[q] == hi[q]) continue;
        for (int j = tid; j < nn[q]; j += VF_THREADS) {
            const uint32_t k = key_at(q, j);
            if (k >= lo[q] && k <= hi[q]) { const int p = atomicAdd(&S.ncand[q], 1); if (p < VF_NCAND) S.cand[q][p] = k; }
        }
    }
    __syncthreads();
    // warp q ranks the candidates of series q: the keys at ranks r and r + 1 inside the bracket
    if (warp < 2) {
        const int q = warp;
        if (nn[q] > 0) {
            uint32_t a = hi[q], b = 0xffffffffu;  // lower / upper middle key; b unknown yet
            bool have_b = false;
            if (lo[q] == hi[q]) {
                have_b = cnt_hi[q] > rank[q] + 1;
                b = hi[q];
            } else {
                const int m = min((int)(cnt_hi[q] - cnt_lo[q]), VF_NCAND);
                const int r = (int)(rank[q] - cnt_lo[q]);
                for (int i = lane; i < m; i += 32) {
                    const uint32_t ki = S.cand[q][i];
                    int pos = 0;
                    for (int j = 0; j < m; j++) { const uint32_t kj = S.cand[q][j]; pos += (kj < ki) || (kj == ki && j < i); }
                    if (pos == r) S.utmp[4 + 2 * q] = ki;
                    if (pos == r + 1) S.utmp[5 + 2 * q] = ki;
                }
                __syncwarp();
                a = S.utmp[4 + 2 * q];
                have_b = (r + 1 < m);
                if (have_b) b = S.utmp[5 + 2 * q];
            }
            if (lane == 0) { S.utmp[4 + 2 * q] = a; S.utmp[5 + 2 * q] = b; S.itmp[q] = have_b ? 1 : 0; }
        }
    }
    __syncthreads();
    for (int q = 0; q < 2; q++) {
        if (nn[q] <= 0) { out[q] = CUDART_NAN_F; continue; }
        const float a = key_f32(S.utmp[4 + 2 * q]);
        if (nn[q] & 1) { out[q] = a; continue; }
        uint32_t up = S.utmp[5 + 2 * q];
        if (!S.itmp[q]) {
            // the upper middle element lies beyond the bracket: smallest key above hi (rare)
            __syncthreads();
            if (tid == 0) S.utmp[3] = 0xffffffffu;
            __syncthreads();
            uint32_t best = 0xffffffffu;
            for (int j = tid; j < nn[q]; j += VF_THREADS) { const uint32_t k = key_at(q, j); if (k > hi[q]) best = min(best, k); }
            best = warp_min_u(best);
            if (lane == 0) atomicMin(&S.utmp[3], best);
            __syncthreads();
            up = S.utmp[3];
            __syncthreads();
        }
        out[q] = __fdiv_rn(__fadd_rn(a, key_f32(up)), 2.0f);
    }
    __syncthreads();
    if (tid < 6) S.cnt[tid] = 0;
    __syncthreads();
}

// ---- the kernel ----------------------------------------------------------------------------------------------------
__host__ __device__ inline size_t vfast_smem_bytes(int win_bytes) {
    return (((size_t)win_bytes + 48 + 15) & ~(size_t)15);  // dynamic part: the window; the scratch is static
}

// one rank task over the window range [a, b) (clipped); returns the task index or -1 if the range is empty
__device__ __forceinline__ int vf_add_rank(VfScratch &S, const VfRead &R, int &nt, int &rot, int a, int b, int k) {
    clip_seg(a, b, R.n);
    const int n = b - a;
    if (n <= 0) return -1;
    const int q = nt++;
    const int nvec = max(((R.s0 + b) >> 3) - ((R.s0 + a + 7) >> 3), 0);
    if (threadIdx.x == 0) {
        VfTask &t = S.task[q];
        t.a = a; t.b = b; t.kind = 0; t.k = k; t.lo = R.kmin; t.hi = R.kmax; t.cnt_hi = n; t.pv = 0; t.med = 0.f;
        t.active = 0; t.sent = R.kmax + 1; t.smin = R.kmin; t.smax = R.kmax;
        vf_geometry(R, t, a, b, rot);
    }
    rot += nvec;
    return q;
}

// value of the order statistics k and k + 1 (if two) of a finished rank task -> codes v0, v1.  CTA-wide (uniform).
__device__ __forceinline__ void vf_rank_pair(const VfRead &R, VfScratch &S, int q, bool two, int &v0, int &v1) {
    const VfTask &t = S.task[q];
    v0 = t.hi;
    v1 = v0;
    const int a = t.a, b = t.b, k = t.k, c = t.cnt_hi;
    if (two && !(c > k + 1)) v1 = vf_neighbour(R, S, a, b, v0, true);
}

// hand the order statistics of range q (finished rank task t; -1: empty range) over to the checks.  CTA-wide (uniform).
__device__ void vf_put_ranks(const VfRead &R, VfScratch &S, int q, int t) {
    int n = 0, v0 = 0, v1 = 0;
    if (t >= 0) {
        bool two;
        n = S.task[t].b - S.task[t].a;
        vc_rank(q, n, two);
        vf_rank_pair(R, S, t, two, v0, v1);
    }
    if (threadIdx.x == 0) { S.st.n[q] = n; S.st.c0[q] = v0; S.st.c1[q] = v1; }
}

struct VfDevOut { float mad; };

// add the deviation-search task of a segment (median known, code bounds [smin, smax] of its samples); returns its
// index or -1
__device__ __forceinline__ int vf_add_mad(VfScratch &S, const VfRead &R, int &nt, int &rot, int a, int b, float med,
                                          int smin, int smax) {
    clip_seg(a, b, R.n);
    const int n = b - a;
    if (n <= 0 || !(med == med)) return -1;
    const int q = nt++;
    int ok = 1;
    int pv = gsb_code_at(med, false, R.coff, R.cscale, &ok);
    pv = min(max(pv, smin), smax + 1);
    const int nvec = max(((R.s0 + b) >> 3) - ((R.s0 + a + 7) >> 3), 0);
    if (threadIdx.x == 0) {
        VfTask &t = S.task[q];
        t.a = a; t.b = b; t.kind = 1; t.k = (n - 1) / 2; t.cnt_hi = -1; t.pv = pv; t.med = med;
        t.smin = smin; t.smax = smax;
        t.lo = 0; t.hi = 0; t.sent = 0;
        t.rlo = 0; t.rhi = smax + 1 - pv; t.llo = 0; t.lhi = pv - smin;
        t.t_best = CUDART_INF_F; t.c_best = -1;
        t.active = 0;
        vf_geometry(R, t, a, b, rot);
    }
    rot += nvec;
    return q;
}

// median of |x - med| from the finished deviation task q.  CTA-wide (uniform).
__device__ float vf_mad_of(const VfRead &R, VfScratch &S, int q) {
    if (q < 0) return CUDART_NAN_F;
    const VfTask t = S.task[q];
    const int n = t.b - t.a, k = t.k, pv = t.pv;
    const float med = t.med;
    const float d0 = t.t_best;  // the last probe that passed is the smallest passing candidate (see vf_update)
    if (n & 1) return d0;
    float d1 = d0;
    if (!(t.c_best > k + 1)) {
        // the next larger deviation: first occupied code beyond the interval [l, r] of the codes deviating <= d0
        int lo = R.kmin, hi = pv;
        while (lo < hi) { const int m = (lo + hi) >> 1; if (vf_dev(R, m, med) <= d0) hi = m; else lo = m + 1; }
        const int l = lo;  // == pv if no left code deviates <= d0
        lo = pv; hi = R.kmax + 1;
        while (lo < hi) { const int m = (lo + hi) >> 1; if (vf_dev(R, m, med) > d0) hi = m; else lo = m + 1; }
        const int r = lo - 1;  // == pv - 1 if no right code deviates <= d0
        const int up = vf_neighbour(R, S, t.a, t.b, r, true);
        const int dn = vf_neighbour(R, S, t.a, t.b, l, false);
        d1 = CUDART_INF_F;
        if (up >= 0) d1 = fminf(d1, vf_dev(R, up, med));
        if (dn >= 0) d1 = fminf(d1, vf_dev(R, dn, med));
    }
    return __fdiv_rn(__fadd_rn(d0, d1), 2.0f);
}

__global__ void __launch_bounds__(VF_THREADS, 4) validate_fast_kernel(VfastArgs A, adb_config cfg) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *winbuf = smem;
    __shared__ VfScratch S;
    __shared__ uint64_t bar_storage;
    uint64_t *bar = &bar_storage;
    const int tid = threadIdx.x;
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    uint32_t phase = 0;

    for (int r = blockIdx.x; r < A.B.n_reads; r += gridDim.x) {
        adb_record *rec = A.out + r;
        // generic-proxy accesses to the window memory of the previous read are ordered before the next bulk copy
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        ReadSrc gsrc;
        if (!vc_read_start(A, r, gsrc)) continue;
        VcIn I;
        if (!vc_inputs(A, cfg, r, gsrc, I)) continue;
        const int size = I.size, a_end = I.a_end;
        // ---- stage the preload window in shared memory (TMA bulk copy) ----
        VfRead R;
        {
            unsigned char *w = cta_stage_window(winbuf, (const unsigned char *)gsrc.i16, size * 2, bar, phase);
            R.W16 = reinterpret_cast<const uint16_t *>(winbuf);
            R.s0 = (int)(w - winbuf) >> 1;
        }
        R.n = size; R.coff = gsrc.coff; R.cscale = gsrc.cscale;
        if (size <= 0) continue;
        vf_minmax(R, S, R.kmin, R.kmax);
        if (R.kmin < 0 || R.kmax >= VF_KEY_LIMIT) continue;  // codes must read as non-negative finite halves
        vc_zero_record(rec);

        // ---- speculative inputs of the checks (SURVEY A.8), all from the staged window ----
        int n_open = 0, op_last = 0;
        if (a_end != 0 && cfg.detect_open_pores) {
            int ok = 1;
            const int c200 = gsb_code_at(200.0f, false, R.coff, R.cscale, &ok);
            n_open = vf_open_pores(R, S, 0, a_end, c200, rec, &op_last);
        }
        const VcGeom G = vc_geometry(cfg, I, n_open, op_last);
        if (G.rr_geom) {
            float rm0, rm1;
            vf_mean_pair(R, S, G.ra, G.ra + G.rlen - cfg.mean_window, cfg.mean_window, rm0, rm1);
            if (tid == 0) { S.st.rm0 = rm0; S.st.rm1 = rm1; }
        }

        // ---- round A: every rank ----
        int nt = 0, rot = 0;
        __syncthreads();
        int tq[VC_NQ];
#pragma unroll
        for (int q = 0; q < VC_NQ; q++) {
            const int n = G.qb[q] - G.qa[q];
            bool two;
            tq[q] = (n > 0) ? vf_add_rank(S, R, nt, rot, G.qa[q], G.qb[q], vc_rank(q, n, two)) : -1;
        }
        if (tid == 0) { S.ntask = nt; S.vtotal = rot; }
        vf_task_bounds(R, S);
        vf_run(R, S);
#pragma unroll
        for (int q = 0; q < VC_NQ; q++) vf_put_ranks(R, S, q, tq[q]);
        __syncthreads();

        // ---- round B: every MAD ----
        const int msrc[4] = {VC_A0, VC_A1, VC_P, VC_R};
        VfTask src[4];  // (the MAD tasks take the places of the rank tasks)
#pragma unroll
        for (int m = 0; m < 4; m++) if (tq[msrc[m]] >= 0) src[m] = S.task[tq[msrc[m]]];
        int dq[4];
        nt = 0; rot = 0;
        __syncthreads();
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const VfTask &t = src[m];
            dq[m] = (tq[msrc[m]] >= 0) ? vf_add_mad(S, R, nt, rot, t.a, t.b, vc_median(S.st, msrc[m], R.coff, R.cscale), t.smin, t.smax) : -1;
        }
        __syncthreads();
        if (tid == 0) { S.ntask = nt; S.vtotal = rot; }
        vf_run(R, S);
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const float mad = vf_mad_of(R, S, dq[m]);
            if (tid == 0) S.st.mad[m] = mad;
        }
        __syncthreads();

        if (tid == 0) {
            vc_small_mean_var(I, reinterpret_cast<const int16_t *>(R.W16) + R.s0, S.st);
            S.out = vc_checks(cfg, I, G, S.st, A.mode, A.cand_followup != 0);
        }
        __syncthreads();
        if (S.out.defer) continue;  // (uniform) validate_kernel redoes this read from scratch
        double pmean[3], pstd[3];
        if (!S.out.exception) {  // partition sums (signal_partitions.py:65-96) while the window is still staged
            int sa[3], sb[3];
            bool on[3];
            for (int p = 0; p < 3; p++) on[p] = vc_partition(I, S.out, p, sa[p], sb[p]);
            vf_mean_std3(R, S, sa, sb, on, pmean, pstd);
        }
        if (!(S.out.valid & ADB_V_OPEN_PORES) || S.out.exception) {
            if (tid < ADB_MAX_OPEN_PORES) rec->open_pores[tid] = 0;  // the scan was speculative
        }
        if (tid == 0) {
            vc_write_spec_record(rec, I, S.st, S.out, pmean, pstd);
            __threadfence();
            A.done[r] = S.out.followup ? 2 : 1;
        }
    }
}

// ---- further poly(A) candidates of the reads whose first one failed (CNN path, combined.py:464-515) ---------------------
// `success` is never reset once a candidate has failed, so the loop of the reference runs to its last non-zero
// candidate whatever happens: the mvs_detect_* values of the record are those of the LAST candidate, the fail reason
// that of the last candidate that failed (scanning backwards from the end until one fails).  Everything else of the
// record -- incl. polya_end = the first candidate and the partition statistics -- stands as validate_fast_kernel wrote
// it.  One evaluation = mean_var_shift_polyA_check (mvs.py:45-158) of one candidate: poly(A) median, p85 - p15, the two
// medians around adapter_end, and the medians of the moving statistics, which are prefixes of the rows the second
// mvs_series_kernel pass computed up to the largest candidate.  A read this kernel cannot settle (series not
// precomputed) goes back to validate_kernel (done = 0).
__global__ void __launch_bounds__(VF_THREADS, 4) validate_cand_kernel(VfastArgs A, adb_config cfg, const int *pending,
                                                                      const int *n_pending) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *winbuf = smem;
    const size_t win_cap = (((size_t)A.win_bytes + 48 + 15) & ~(size_t)15);
    __shared__ VfScratch S;
    __shared__ uint64_t bar_storage;
    uint64_t *bar = &bar_storage;
    const int tid = threadIdx.x;
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    uint32_t phase = 0;
    const int n_list = *n_pending;
    const int msw = cfg.median_shift_window;
    for (int li = blockIdx.x; li < n_list; li += gridDim.x) {
        const int r = pending[li];
        if (A.done[r] != 2) continue;
        adb_record *rec = A.out + r;
        const ReadSrc gsrc = make_src(A.B, r);
        const int size = gsrc.n;
        const int *g = A.given + (size_t)r * A.given_stride;
        const int a_end = g[0];
        const int n_topk = A.ntopk_per_read ? A.ntopk_per_read[r] : A.given_ntopk;
        int n_eval = 0;
        while (n_eval < n_topk && g[1 + n_eval] != 0) n_eval++;
        const long long po = A.pre_off ? A.pre_off[r] : -1;
        const bool have_rows = po >= 0 && A.pre_meta[2 * r] == a_end;
        const int row_pe = have_rows ? A.pre_meta[2 * r + 1] : 0;
        const float medA0 = *reinterpret_cast<const float *>(rec->_reserved);
        double mr[2];
        vc_pa_mean_bounds(cfg, medA0, mr);  // (empty bounds raised in validate_fast_kernel: no follow-up)
        double last_v[5] = {0, 0, 0, 0, 0};
        int fail = rec->fail_code, fail_mask = rec->mvs_fail_mask;  // the first candidate's, unless a later one failed
        bool bail = false, fail_known = false;
        for (int t = n_eval - 1; t >= 1 && !fail_known && !bail; t--) {
            const int pe = g[1 + t];
            double v[5] = {0, 0, 0, 0, 0};
            bool ok = false;
            const bool geom = !(pe == 0 || a_end == 0 || pe < a_end || pe - a_end <= 2) && !(size < a_end + msw);
            if (geom) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncthreads();
                VfRead R;
                {
                    unsigned char *w = cta_stage_window(winbuf, (const unsigned char *)gsrc.i16, size * 2, bar, phase);
                    R.W16 = reinterpret_cast<const uint16_t *>(winbuf);
                    R.s0 = (int)(w - winbuf) >> 1;
                }
                R.n = size; R.coff = gsrc.coff; R.cscale = gsrc.cscale;
                vf_minmax(R, S, R.kmin, R.kmax);  // (the first pass has verified 0 <= code < VF_KEY_LIMIT)
                int pa_ = a_end, pb_ = pe;
                clip_seg(pa_, pb_, size);
                const int nP = pb_ - pa_;
                const bool win_var = !(pe - a_end <= cfg.pA_var_window + 2), win_mean = !(pe - a_end <= cfg.pA_mean_window + 2);
                const int nv = win_var ? nP - (cfg.pA_var_window - 1) : 0, nm = win_mean ? nP - (cfg.pA_mean_window - 1) : 0;
                if ((win_var || win_mean) && !(have_rows && row_pe >= pe)) { bail = true; break; }
                const bool big = (size_t)(((max(nv, 0) + 3) & ~3) + max(nm, 0)) * 4 > win_cap;  // series beyond the window memory
                int nt = 0, rot = 0;
                __syncthreads();
                const int cq[5] = {VC_P, VC_P15, VC_P85, VC_AF, VC_BF};
                const int ca[5] = {a_end, a_end, a_end, a_end, max(a_end - msw, 0)};
                const int cb[5] = {pe, pe, pe, min(a_end + msw, size), a_end};
                int tq[5];
#pragma unroll
                for (int c = 0; c < 5; c++) {
                    int a = ca[c], b = cb[c];
                    clip_seg(a, b, size);
                    bool two;
                    tq[c] = (b > a) ? vf_add_rank(S, R, nt, rot, a, b, vc_rank(cq[c], b - a, two)) : -1;
                }
                if (tid == 0) { S.ntask = nt; S.vtotal = rot; }
                vf_task_bounds(R, S);
                vf_run(R, S);
#pragma unroll
                for (int c = 0; c < 5; c++) vf_put_ranks(R, S, cq[c], tq[c]);
                if ((!win_var || !win_mean) && tid == 0) {
                    const int16_t *p = reinterpret_cast<const int16_t *>(R.W16) + R.s0 + pa_;
                    auto x = [&](int i) { return gsb_pa(p[i], R.coff, R.cscale); };
                    S.st.small_mean = np_mean_f32(x, nP);
                    S.st.small_var = np_var_f32(x, nP, S.st.small_mean);
                }
                __syncthreads();
                float smed[2] = {0.f, 0.f};
                if (big) vf_series_medians<false>(S, A.pre_var + po, max(nv, 0), A.pre_mean + po, max(nm, 0), (uint32_t *)winbuf, smed);
                else if (nv > 0 || nm > 0) vf_series_medians<true>(S, A.pre_var + po, max(nv, 0), A.pre_mean + po, max(nm, 0), (uint32_t *)winbuf, smed);
                v[0] = (double)(win_mean ? smed[1] : S.st.small_mean);
                v[1] = (double)(win_var ? smed[0] : S.st.small_var);
                v[2] = (double)vc_median(S.st, VC_P, R.coff, R.cscale);
                v[3] = vc_local_range(S.st, VC_P15, VC_P85, R.coff, R.cscale);
                v[4] = (double)__fsub_rn(vc_median(S.st, VC_AF, R.coff, R.cscale), vc_median(S.st, VC_BF, R.coff, R.cscale));
                const int mask = vc_mvs_mask(cfg, v, mr);
                ok = (mask == 0);
                if (!ok) {
                    vc_mvs_fail(v[0], mask, fail, fail_mask);
                    fail_known = true;
                }
            } else {  // the early return of mean_var_shift_polyA_check: zeros, "not enough signal"
                fail = ADB_FAIL_MVS_NOT_ENOUGH; fail_mask = 0;
                fail_known = true;
            }
            if (t == n_eval - 1) for (int i = 0; i < 5; i++) last_v[i] = v[i];
        }
        __syncthreads();
        if (tid == 0) {
            if (bail) {
                A.done[r] = 0;  // validate_kernel redoes the read from scratch
            } else {
                for (int i = 0; i < 5; i++) rec->mvs[i] = last_v[i];
                rec->fail_code = fail;
                rec->mvs_fail_mask = fail_mask;
                for (int i = 0; i < 8; i++) rec->_reserved[i] = 0;
                __threadfence();
                A.done[r] = 1;
            }
        }
    }
}
