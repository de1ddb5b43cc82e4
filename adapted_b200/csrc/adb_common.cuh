// Shared device helpers for the adapted_b200 kernels (sm_100a).
//
// Arithmetic contract (SURVEY.md A.1/A.2): everything that feeds an integer decision reproduces the
// reference's association order with individually rounded IEEE operations -- the file is compiled with
// -fmad=false and uses the __f*_rn / __d*_rn intrinsics where the order matters.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/adapted_b200.h"

#define ADB_WARP 32
#define ADB_FULL 0xffffffffu

// ---------------------------------------------------------------------------------------------------------
// signal source of one read: calibrated float32 or raw int16 + calibration
// ---------------------------------------------------------------------------------------------------------
struct ReadSrc {
    const float *f32;     // != nullptr for ADB_SIG_F32
    const int16_t *i16;   // != nullptr for ADB_SIG_I16
    int n;                // valid samples = min(full_len, m)
    float coff, cscale;   // pA = (adc + coff) * cscale, float32 ops

    // plain loads: the pointers may address global memory or a window staged in shared memory
    __device__ __forceinline__ float pa(int j) const {
        if (f32) return f32[j];
        return __fmul_rn(__fadd_rn((float)i16[j], coff), cscale);
    }
};

struct BatchDev {  // device-side view of adb_batch
    const void *signal;
    int sig_type, n_reads, m, batch_size;
    const int64_t *offsets;
    const int32_t *full_lens;
    const float *calib_offset, *calib_scale;
};

__device__ __forceinline__ ReadSrc make_src(const BatchDev &b, int r) {
    ReadSrc s;
    int fl = b.full_lens[r];
    if (b.sig_type == ADB_SIG_F32) {
        s.f32 = (const float *)b.signal + (size_t)r * b.m;
        s.i16 = nullptr;
        s.n = min(max(fl, 0), b.m);
        s.coff = 0.f;
        s.cscale = 1.f;
    } else {
        int64_t o0 = b.offsets[r], o1 = b.offsets[r + 1];
        s.f32 = nullptr;
        s.i16 = (const int16_t *)b.signal + o0;
        s.n = (int)min((int64_t)b.m, o1 - o0);
        s.coff = b.calib_offset[r];
        s.cscale = b.calib_scale[r];
    }
    return s;
}

// ---------------------------------------------------------------------------------------------------------
// TMA bulk copy global -> shared (cp.async.bulk, SASS UBLKCP) completing on an mbarrier
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t phase) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    while (!mbar_try_wait(bar, phase)) {
    }
}
// dst (shared) and src (global) 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Stage `nbytes` bytes starting at the (arbitrarily aligned) global address `src` into shared memory so that the
// shared copy has the same 16-byte phase as the source: returns the shared address of src[0].  `buf` is 16-byte
// aligned with room for nbytes + 32.  The 16-byte aligned body goes through the TMA bulk engine (one thread issues,
// everybody waits on the mbarrier), the unaligned head / tail with ordinary loads.  CTA-wide.
__device__ unsigned char *cta_stage_window(unsigned char *buf, const unsigned char *src, int nbytes, uint64_t *bar,
                                           uint32_t &phase) {
    const int shift = (int)((uintptr_t)src & 15);
    unsigned char *dst0 = buf + shift;  // dst0 == shared image of src[0]
    if (nbytes <= 0) return dst0;
    const unsigned char *body_src = src + ((16 - shift) & 15);
    const int head = (int)(body_src - src);
    int body = nbytes - head;
    if (body < 0) body = 0;
    body &= ~15;
    const int tail0 = head + body;
    if (threadIdx.x == 0 && body > 0) {
        mbar_expect_tx(bar, (uint32_t)body);
        const int CH = 16384;
        for (int o = 0; o < body; o += CH)
            tma_bulk_g2s(dst0 + head + o, body_src + o, (uint32_t)min(CH, body - o), bar);
    }
    for (int i = threadIdx.x; i < min(head, nbytes); i += blockDim.x) dst0[i] = src[i];
    for (int i = tail0 + threadIdx.x; i < nbytes; i += blockDim.x) dst0[i] = src[i];
    if (body > 0) {
        mbar_wait(bar, phase);
        phase ^= 1;
    }
    __syncthreads();
    return dst0;
}

// ---------------------------------------------------------------------------------------------------------
// order-preserving keys
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f32_key(float v) {
    uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_f32(uint32_t k) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}

// ---------------------------------------------------------------------------------------------------------
// warp / block reductions
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(ADB_FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(ADB_FULL, v, o);
    return v;
}
__device__ __forceinline__ uint32_t warp_min_u(uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(ADB_FULL, v, o));
    return v;
}
__device__ __forceinline__ uint32_t warp_max_u(uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(ADB_FULL, v, o));
    return v;
}

// python slice clipping of [a, b) to [0, size)
__device__ __forceinline__ void clip_seg(int &a, int &b, int size) {
    a = min(max(a, 0), size);
    b = min(max(b, 0), size);
    if (b < a) b = a;
}

// in_range of adapted/detect/utils.py:16-26 on doubles (NaN -> false)
__device__ __forceinline__ bool in_range_d(double v, const double r[2]) { return r[0] <= v && v <= r[1]; }

// ---------------------------------------------------------------------------------------------------------
// numpy pairwise summation (numpy/_core/src/umath/loops_utils.h.src) -- exact association order
// ---------------------------------------------------------------------------------------------------------
// float32, n <= 128 (one leaf).  F: float(int)
template <class F>
__device__ __forceinline__ float np_sum_f32_leaf(F f, int n) {
    if (n < 8) {
        float res = 0.f;
        for (int i = 0; i < n; i++) res = __fadd_rn(res, f(i));
        return res;
    }
    float r0 = f(0), r1 = f(1), r2 = f(2), r3 = f(3), r4 = f(4), r5 = f(5), r6 = f(6), r7 = f(7);
    int i;
    for (i = 8; i < n - (n % 8); i += 8) {
        r0 = __fadd_rn(r0, f(i));
        r1 = __fadd_rn(r1, f(i + 1));
        r2 = __fadd_rn(r2, f(i + 2));
        r3 = __fadd_rn(r3, f(i + 3));
        r4 = __fadd_rn(r4, f(i + 4));
        r5 = __fadd_rn(r5, f(i + 5));
        r6 = __fadd_rn(r6, f(i + 6));
        r7 = __fadd_rn(r7, f(i + 7));
    }
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r0, r1), __fadd_rn(r2, r3)),
                          __fadd_rn(__fadd_rn(r4, r5), __fadd_rn(r6, r7)));
    for (; i < n; i++) res = __fadd_rn(res, f(i));
    return res;
}

// float32, any n, executed by ONE thread (explicit stack instead of recursion).
template <class F>
__device__ float np_sum_f32(F f, int n) {
    // iterative post-order evaluation of: S(lo,n) = n<=128 ? leaf : S(lo,n2) + S(lo+n2,n-n2)
    int lo_stack[24], n_stack[24];
    float val_stack[24];
    unsigned char state[24];
    int sp = 0, vp = 0;
    lo_stack[0] = 0; n_stack[0] = n; state[0] = 0; sp = 1;
    while (sp > 0) {
        int lo = lo_stack[sp - 1], nn = n_stack[sp - 1];
        if (nn <= 128) {
            val_stack[vp++] = np_sum_f32_leaf([&](int i) { return f(lo + i); }, nn);
            sp--;
        } else if (state[sp - 1] == 0) {
            int n2 = nn / 2; n2 -= n2 % 8;
            state[sp - 1] = 1;
            // push right first so that left is evaluated first
            lo_stack[sp] = lo + n2; n_stack[sp] = nn - n2; state[sp] = 0; sp++;
            lo_stack[sp] = lo; n_stack[sp] = n2; state[sp] = 0; sp++;
        } else {
            float right = val_stack[--vp], left = val_stack[--vp];
            val_stack[vp++] = __fadd_rn(left, right);
            sp--;
        }
    }
    return val_stack[0];
}

template <class F>
__device__ __forceinline__ double np_sum_f64_leaf(F f, int n) {
    if (n < 8) {
        double res = 0.;
        for (int i = 0; i < n; i++) res = __dadd_rn(res, f(i));
        return res;
    }
    double r0 = f(0), r1 = f(1), r2 = f(2), r3 = f(3), r4 = f(4), r5 = f(5), r6 = f(6), r7 = f(7);
    int i;
    for (i = 8; i < n - (n % 8); i += 8) {
        r0 = __dadd_rn(r0, f(i));
        r1 = __dadd_rn(r1, f(i + 1));
        r2 = __dadd_rn(r2, f(i + 2));
        r3 = __dadd_rn(r3, f(i + 3));
        r4 = __dadd_rn(r4, f(i + 4));
        r5 = __dadd_rn(r5, f(i + 5));
        r6 = __dadd_rn(r6, f(i + 6));
        r7 = __dadd_rn(r7, f(i + 7));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r0, r1), __dadd_rn(r2, r3)),
                           __dadd_rn(__dadd_rn(r4, r5), __dadd_rn(r6, r7)));
    for (; i < n; i++) res = __dadd_rn(res, f(i));
    return res;
}

// float64, any n, ONE thread
template <class F>
__device__ double np_sum_f64(F f, int n) {
    int lo_stack[24], n_stack[24];
    double val_stack[24];
    unsigned char state[24];
    int sp = 0, vp = 0;
    lo_stack[0] = 0; n_stack[0] = n; state[0] = 0; sp = 1;
    while (sp > 0) {
        int lo = lo_stack[sp - 1], nn = n_stack[sp - 1];
        if (nn <= 128) {
            val_stack[vp++] = np_sum_f64_leaf([&](int i) { return f(lo + i); }, nn);
            sp--;
        } else if (state[sp - 1] == 0) {
            int n2 = nn / 2; n2 -= n2 % 8;
            state[sp - 1] = 1;
            lo_stack[sp] = lo + n2; n_stack[sp] = nn - n2; state[sp] = 0; sp++;
            lo_stack[sp] = lo; n_stack[sp] = n2; state[sp] = 0; sp++;
        } else {
            double right = val_stack[--vp], left = val_stack[--vp];
            val_stack[vp++] = __dadd_rn(left, right);
            sp--;
        }
    }
    return val_stack[0];
}

// np.percentile(method="linear") interpolation between two float32 order statistics
// (numpy/lib/_function_base_impl.py _lerp): the difference is taken in the input dtype (float32), the
// interpolation in float64.  g = fractional part of (n-1)*q.
__device__ __forceinline__ double np_lerp_f32(float a, float b, double g) {
    double d = (double)__fsub_rn(b, a);
    double r = __dadd_rn((double)a, __dmul_rn(d, g));
    if (g >= 0.5) r = __dsub_rn((double)b, __dmul_rn(d, __dsub_rn(1.0, g)));
    return r;
}
