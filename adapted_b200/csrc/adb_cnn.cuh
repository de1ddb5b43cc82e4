// CNN primary boundaries (cnn_detect_boundaries, adapted/detect/cnn.py:16-201).
//
//   cnn_prep_kernel     prepare_data (cnn.py:70-82): mean-pool downscale of batch[:, min_obs_adapter:], per-read
//                       nanmedian / MAD normalisation (no clipping), nan_to_num(-5).
//   cnn_conv64_tc_kernel (adb_cnn_tc.cuh)  layers 2 and 3 (Conv1d 64->64, k=7, pad 3, ReLU) on the tcgen05 tensor
//                       cores; layer 1 fused into layer 2's operand build, layer 4 into layer 3's epilogue.
//   cnn_conv64_kernel   the same two layers as a register-tiled implicit GEMM on the FP32 pipe: recomputes the reads the
//                       tensor-core kernels flag (values outside their fp16 split), or every read with the
//                       "cnn_fp32_pipe" option; layer 1 (Conv1d 1->64, k=7, stride 3, pad 3, ReLU) fused into layer 2.
//   cnn_convT_kernel    layer 4 (ConvTranspose1d 64->2, k=7, stride 3, pad 3) -> scores [N, 2, L_out] for that path.
//   cnn_mask_kernel / cnn_peaks_* / cnn_topk_kernel / cnn_shift_kernel
//                       cnn_predict's post-processing (cnn.py:117-160): adapter argmax, masking, poly(A) argmax,
//                       find_peaks(flattened scores, distance=5) with its cross-read plateau / distance coupling,
//                       per-read top-k by height, and the "groups shift up when a read has no peak" behaviour
//                       (SURVEY.md A.6), then cnn_detect's coordinate mapping (cnn.py:173-179).
//
// Precision: the reference is float32 (torch CPU, oneDNN's summation order, not reproducible bit for bit); the contract
// is "boundaries within +-1 downscaled step" (north_star).  The FP32-pipe kernels accumulate every product with fmaf in
// float32; the tensor-core kernels keep ~22 bits per operand (fp16 hi / lo split) and accumulate in float32.
#pragma once
#include "adb_series_median.cuh"
#include <cuda_fp16.h>
#include <float.h>

#include "adb_common.cuh"
#include "adb_ctx.cuh"
#include "adb_select.cuh"
#include <algorithm>

#define ADB_CNN_NPARAMS 58882
#define CNN_C 64
#define CNN_K 7
#define CNN_SCORE_EXCL (-5.0f)
// offsets into the flat state dict (0.weight, 0.bias, 2.weight, 2.bias, 4.weight, 4.bias, 6.weight, 6.bias)
#define CNN_W1 0
#define CNN_B1 (CNN_W1 + 64 * 7)
#define CNN_W2 (CNN_B1 + 64)
#define CNN_B2 (CNN_W2 + 64 * 64 * 7)
#define CNN_W3 (CNN_B2 + 64)
#define CNN_B3 (CNN_W3 + 64 * 64 * 7)
#define CNN_W4 (CNN_B3 + 64)
#define CNN_B4 (CNN_W4 + 64 * 2 * 7)

#define CNN_TILE 96       // output positions per tile of the 64->64 convolutions
#define CNN_TILE_IN 104   // input tile row stride (CNN_TILE + 6, padded)
#define CNN_THREADS 192   // 8 output-channel groups x 24 position groups; each thread: 8 channels x 4 positions

// ---- prepare_data ----------------------------------------------------------------------------------------------
struct SmemKeys {
    const float *p;
    __device__ __forceinline__ uint32_t operator()(int j) const { return f32_key(p[j]); }
};
struct SmemDevKeys {
    const float *p;
    float med;
    __device__ __forceinline__ uint32_t operator()(int j) const { return f32_key(fabsf(__fsub_rn(p[j], med))); }
};
struct KeyF32Id {
    __device__ __forceinline__ float operator()(uint32_t k) const { return key_f32(k); }
};

template <class F>
__device__ __forceinline__ float cnn_block_mean(F f, int factor) {
    return __fdiv_rn(np_sum_f32_leaf(f, factor), (float)factor);
}

// x[r][0..L) ; L = ceil((m - A0) / f).  One CTA (256 threads) per read; dynamic smem = L floats + select scratch.
__global__ void __launch_bounds__(256) cnn_prep_kernel(BatchDev B, int A0, int f, int L, float *x) {
    extern __shared__ __align__(16) unsigned char smem[];
    float *ds = (float *)smem;
    unsigned char *scr = smem + (((size_t)L * 4 + 15) & ~(size_t)15);
    SelScratch S = sel_scratch_from(scr);
    uint32_t *kbuf = (uint32_t *)(scr + ((ADB_SEL_SMEM_BYTES + 15) & ~15));
    const int r = blockIdx.x;
    const ReadSrc src = make_src(B, r);
    // leading NaN-free bins (the rest of the row is NaN: NaN padding of the minibatch matrix, file_proc.py:172-174)
    int nv;
    {
        const int span = B.m - A0;
        if (span <= 0) nv = 0;
        else if (src.n >= B.m) nv = L;
        else nv = (src.n > A0) ? (src.n - A0) / f : 0;
        nv = min(nv, L);
    }
    for (int b = threadIdx.x; b < nv; b += blockDim.x) {
        const int j0 = A0 + b * f;
        ds[b] = cnn_block_mean([&](int k) { const int j = j0 + k; return (j < B.m) ? src.pa(j) : 0.0f; }, f);
    }
    __syncthreads();
    float med = CUDART_NAN_F, mad = CUDART_NAN_F;
    if (nv > 0) {
        uint32_t kmin, kmax;
        SmemKeys K{ds};
        cta_key_minmax(K, nv, kmin, kmax, S);
        med = cta_median_keys(K, KeyF32Id(), nv, kmin, kmax, S, kbuf);
        SmemDevKeys D{ds, med};
        const float dmax = fmaxf(fabsf(__fsub_rn(key_f32(kmax), med)), fabsf(__fsub_rn(key_f32(kmin), med)));
        mad = cta_median_keys(D, KeyF32Id(), nv, f32_key(0.0f), f32_key(dmax), S, kbuf);
    }
    float *xr = x + (size_t)r * L;
    for (int b = threadIdx.x; b < L; b += blockDim.x) {
        float v = CNN_SCORE_EXCL;
        if (b < nv) {
            v = __fdiv_rn(__fsub_rn(ds[b], med), mad);
            if (!(v == v)) v = CNN_SCORE_EXCL;          // torch.nan_to_num(nan=-5)
            else if (v == CUDART_INF_F) v = FLT_MAX;
            else if (v == -CUDART_INF_F) v = -FLT_MAX;
        }
        xr[b] = v;
    }
}

// The same, one WARP per read (int16 sources): the downscaled row (1650 bins for RNA004) and its ordered keys live in
// the warp's slice of shared memory, median and MAD are two warp-level selects (warp_select2, adb_series_median.cuh:
// sampled opening bracket, bisection with warp counts, the last 64 keys ranked directly) -- no CTA barrier, 16 reads in
// flight per SM.  Exact order statistics: identical to cnn_prep_kernel.
#define PREP_WARPS 4
#define PREP_CHUNK_BINS 320   // bins per staged chunk: 320 x downscale factor 10 x 2 B = 6400 B <= the warp's key area
__host__ __device__ inline size_t cnn_prep_warp_smem(int L) { return (size_t)PREP_WARPS * (2 * ((L + 3) & ~3) + SM_NCAND + 4) * 4; }
__global__ void __launch_bounds__(PREP_WARPS * 32) cnn_prep_warp_kernel(BatchDev B, int A0, int f, int L, float *x) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int Lp = (L + 3) & ~3;
    float *ds = (float *)smem + (size_t)warp * (2 * Lp + SM_NCAND + 4);
    uint32_t *keys = (uint32_t *)(ds + Lp), *cand = keys + Lp;
    __shared__ uint64_t pbar[PREP_WARPS];
    if (threadIdx.x < PREP_WARPS) mbar_init(&pbar[threadIdx.x], 1);
    __syncthreads();
    uint32_t pphase = 0;
    for (int r = blockIdx.x * PREP_WARPS + warp; r < B.n_reads; r += gridDim.x * PREP_WARPS) {
        const ReadSrc src = make_src(B, r);
        int nv;
        {
            const int span = B.m - A0;
            if (span <= 0) nv = 0;
            else if (src.n >= B.m) nv = L;
            else nv = (src.n > A0) ? (src.n - A0) / f : 0;
            nv = min(nv, L);
        }
        const int nvp = (nv + 3) & ~3;
        if (lane == 0) {  // the window of this warp's next read travels to L2 while this one is worked on
            const int rn = r + gridDim.x * PREP_WARPS;
            if (rn < B.n_reads) {
                const ReadSrc nx = make_src(B, rn);
                if (nx.i16 != nullptr && nx.n > A0 + 16) {
                    const uintptr_t p0 = ((uintptr_t)(nx.i16 + A0) + 15) & ~(uintptr_t)15;
                    const uint32_t nbytes = (uint32_t)(((uintptr_t)(nx.i16 + min(nx.n, B.m)) - p0) & ~(uintptr_t)15);
                    if (nbytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p0), "r"(nbytes) : "memory");
                }
            }
        }
        uint32_t mn = 0xffffffffu, mx = 0u;
        // The raw samples of the NaN-free bins travel to the warp's slice in chunks of PREP_CHUNK_BINS bins (the 16-byte
        // aligned interior of a chunk by one TMA bulk copy, the few samples around it by ordinary loads; the `keys` area
        // is free until the row is complete), the block means are formed from shared memory: ten conflict-free 2-byte
        // loads per bin instead of ten strided global loads.
        {
            int16_t *raw = reinterpret_cast<int16_t *>(keys);
            const int16_t *g0 = src.i16 + A0;                     // first sample of bin 0
            const int cbins = min(PREP_CHUNK_BINS, (Lp * 4 - 16) / (2 * f));  // bins per chunk that fit the key area
            const int n_have = min(src.n, B.m) - A0;              // samples that exist behind A0
            for (int b0 = 0; b0 < nv; b0 += cbins) {
                const int nbin = min(cbins, nv - b0), ns = min(nbin * f, n_have - b0 * f);
                const int16_t *gs = g0 + (size_t)b0 * f;          // first sample of the chunk
                const int shift = (int)(((uintptr_t)gs & 15) >> 1);  // the chunk sits at raw[shift ...): same 16-byte phase
                const int head = min((8 - shift) & 7, ns);         // samples before the aligned interior
                const int body = (ns - head) & ~7;                 // samples of the interior (a multiple of 8)
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0 && body > 0) {
                    mbar_expect_tx(&pbar[warp], (uint32_t)body * 2);
                    tma_bulk_g2s(raw + shift + head, gs + head, (uint32_t)body * 2, &pbar[warp]);
                }
                for (int i = lane; i < head; i += 32) raw[shift + i] = gs[i];
                for (int i = head + body + lane; i < ns; i += 32) raw[shift + i] = gs[i];
                if (body > 0) { mbar_wait(&pbar[warp], pphase); pphase ^= 1; }
                __syncwarp();
                const int16_t *rs = raw + shift;
                for (int b = lane; b < nbin; b += 32) {
                    const int16_t *p = rs + b * f;
                    const int left = ns - b * f;                   // staged samples from the bin's start (< f: ragged last bin)
                    const float v = cnn_block_mean([&](int k) { return (k < left) ? __fmul_rn(__fadd_rn((float)(int)p[k], src.coff), src.cscale) : 0.0f; }, f);
                    ds[b0 + b] = v;
                    const uint32_t k0 = f32_key(v);
                    mn = min(mn, k0); mx = max(mx, k0);
                }
                __syncwarp();
            }
            for (int b = lane; b < nv; b += 32) keys[b] = f32_key(ds[b]);
        }
        if (lane < nvp - nv) keys[nv + lane] = 0xffffffffu;  // pad to full vectors with keys above every rank looked for
        mn = __reduce_min_sync(ADB_FULL, mn);
        mx = __reduce_max_sync(ADB_FULL, mx);
        __syncwarp();
        float med = CUDART_NAN_F, mad = CUDART_NAN_F;
        if (nv > 0) {
            const SmKeys K{reinterpret_cast<const uint4 *>(keys), nullptr};
            const unsigned rank = (unsigned)(nv - 1) >> 1;
            uint32_t a, b2;
            bool hb;
            warp_select2(K, nvp >> 2, 0u, false, nvp, rank, mn, mx, cand, a, b2, hb);
            med = (nv & 1) ? key_f32(a) : __fdiv_rn(__fadd_rn(key_f32(a), key_f32(b2)), 2.0f);
            __syncwarp();
            mn = 0xffffffffu; mx = 0u;
            for (int b = lane; b < nv; b += 32) {
                const uint32_t k = f32_key(fabsf(__fsub_rn(ds[b], med)));
                keys[b] = k;
                mn = min(mn, k); mx = max(mx, k);
            }
            mn = __reduce_min_sync(ADB_FULL, mn);
            mx = __reduce_max_sync(ADB_FULL, mx);
            __syncwarp();
            warp_select2(K, nvp >> 2, 0u, false, nvp, rank, mn, mx, cand, a, b2, hb);
            mad = (nv & 1) ? key_f32(a) : __fdiv_rn(__fadd_rn(key_f32(a), key_f32(b2)), 2.0f);
        }
        float *xr = x + (size_t)r * L;
        for (int b = lane; b < L; b += 32) {
            float v = CNN_SCORE_EXCL;
            if (b < nv) {
                v = __fdiv_rn(__fsub_rn(ds[b], med), mad);
                if (!(v == v)) v = CNN_SCORE_EXCL;          // torch.nan_to_num(nan=-5)
                else if (v == CUDART_INF_F) v = FLT_MAX;
                else if (v == -CUDART_INF_F) v = -FLT_MAX;
            }
            xr[b] = v;
        }
        __syncwarp();
    }
}

// ---- weights: torch layout w[co][ci][k] -> [ci][k][co] so that a thread's 8 output channels are contiguous ---------
__global__ void cnn_pack_weights_kernel(const float *w, float *packed /* 2 x [64][7][64] */) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * CNN_C * CNN_K * CNN_C) return;
    const int layer = i / (CNN_C * CNN_K * CNN_C);
    const int rem = i % (CNN_C * CNN_K * CNN_C);
    const int ci = rem / (CNN_K * CNN_C), k = (rem / CNN_C) % CNN_K, co = rem % CNN_C;
    const float *src = w + (layer == 0 ? CNN_W2 : CNN_W3);
    packed[i] = src[(co * CNN_C + ci) * CNN_K + k];
}

// ---- Conv1d(64 -> 64, k = 7, pad 3) + ReLU ------------------------------------------------------------------------------
// in  : FUSE_L1 ? x [N][Lx] : act [N][64][LP]        out : act [N][64][LP]   (LP = padded row length, multiple of 4)
// Persistent CTAs; the 114.7 KB of packed weights stay in shared memory for the CTA's whole life.
// `only` (optional, [n_reads]): process just the reads flagged there (the reads the tensor-core kernel could not
// represent in its fp16 split, adb_cnn_tc.cuh).
template <bool FUSE_L1>
__global__ void __launch_bounds__(CNN_THREADS, 1) cnn_conv64_kernel(const float *in, float *out, const float *packed_w,
                                                                   const float *bias, const float *w1, const float *b1,
                                                                   int n_reads, int Lx, int L1, int LP, const int *only) {
    if (only) {  // nothing flagged (only[-1] == 0) or nothing flagged for this CTA: leave before the weights are loaded
        if (only[-1] == 0) return;
        const int tiles_per_read = (L1 + CNN_TILE - 1) / CNN_TILE, n_tiles = n_reads * tiles_per_read;
        bool mine = false;
        for (int tile = blockIdx.x; tile < n_tiles && !mine; tile += gridDim.x) mine = only[tile / tiles_per_read] != 0;
        if (!__syncthreads_or(mine)) return;
    }
    extern __shared__ __align__(16) float sm[];
    float *Ws = sm;                                   // [64][7][64]
    float *Is = Ws + CNN_C * CNN_K * CNN_C;           // [64][CNN_TILE_IN]
    float *Xs = Is + CNN_C * CNN_TILE_IN;             // FUSE_L1: x window, 3*(CNN_TILE+6)+8 floats
    float *W1s = Xs + 3 * (CNN_TILE + 6) + 8;         // [64][7] + [64]
    for (int i = threadIdx.x; i < CNN_C * CNN_K * CNN_C; i += blockDim.x) Ws[i] = packed_w[i];
    if (FUSE_L1) {
        for (int i = threadIdx.x; i < CNN_C * CNN_K; i += blockDim.x) W1s[i] = w1[i];
        for (int i = threadIdx.x; i < CNN_C; i += blockDim.x) W1s[CNN_C * CNN_K + i] = b1[i];
    }
    __syncthreads();
    const int tiles_per_read = (L1 + CNN_TILE - 1) / CNN_TILE;
    const int n_tiles = n_reads * tiles_per_read;
    const int cg = threadIdx.x / 24, tg = threadIdx.x % 24;
    const int co0 = cg * 8, tp = tg * 4;
    float bv[8];
#pragma unroll
    for (int c = 0; c < 8; c++) bv[c] = bias[co0 + c];
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int r = tile / tiles_per_read, t0 = (tile % tiles_per_read) * CNN_TILE;
        if (only && !only[r]) continue;
        __syncthreads();
        if (FUSE_L1) {
            // x window needed by act1 positions [t0-3, t0+CNN_TILE+3): x[3p-3 .. 3p+3]
            const float *xr = in + (size_t)r * Lx;
            const int x0 = 3 * (t0 - 3) - 3, nx = 3 * (CNN_TILE + 6) + 6;
            for (int i = threadIdx.x; i < nx; i += blockDim.x) {
                const int j = x0 + i;
                Xs[i] = (j >= 0 && j < Lx) ? xr[j] : 0.0f;
            }
            __syncthreads();
            for (int i = threadIdx.x; i < CNN_C * (CNN_TILE + 6); i += blockDim.x) {
                const int ci = i / (CNN_TILE + 6), q = i % (CNN_TILE + 6);
                const int p = t0 - 3 + q;
                float v = 0.0f;  // zero padding of layer 2's input outside [0, L1)
                if (p >= 0 && p < L1) {
                    float a = W1s[CNN_C * CNN_K + ci];
#pragma unroll
                    for (int k = 0; k < CNN_K; k++) a = fmaf(W1s[ci * CNN_K + k], Xs[3 * q + k], a);
                    v = fmaxf(a, 0.0f);
                }
                Is[ci * CNN_TILE_IN + q] = v;
            }
        } else {
            const float *ar = in + (size_t)r * CNN_C * LP;
            for (int i = threadIdx.x; i < CNN_C * (CNN_TILE + 6); i += blockDim.x) {
                const int ci = i / (CNN_TILE + 6), q = i % (CNN_TILE + 6);
                const int p = t0 - 3 + q;
                Is[ci * CNN_TILE_IN + q] = (p >= 0 && p < L1) ? ar[(size_t)ci * LP + p] : 0.0f;
            }
        }
        __syncthreads();
        float acc[8][4];
#pragma unroll
        for (int c = 0; c < 8; c++)
#pragma unroll
            for (int t = 0; t < 4; t++) acc[c][t] = bv[c];
#pragma unroll 2
        for (int ci = 0; ci < CNN_C; ci++) {
            float iv[10];
            const float *ip = Is + ci * CNN_TILE_IN + tp;
#pragma unroll
            for (int q = 0; q < 10; q++) iv[q] = ip[q];
            const float *wp = Ws + ci * CNN_K * CNN_C + co0;
#pragma unroll
            for (int k = 0; k < CNN_K; k++) {
                const float4 wa = *(const float4 *)(wp + k * CNN_C);
                const float4 wb = *(const float4 *)(wp + k * CNN_C + 4);
                const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                for (int c = 0; c < 8; c++)
#pragma unroll
                    for (int t = 0; t < 4; t++) acc[c][t] = fmaf(wv[c], iv[t + k], acc[c][t]);
            }
        }
        float *orow = out + (size_t)r * CNN_C * LP;
        const int p0 = t0 + tp;
        if (p0 < L1) {
#pragma unroll
            for (int c = 0; c < 8; c++) {
                float4 v = make_float4(fmaxf(acc[c][0], 0.f), fmaxf(acc[c][1], 0.f), fmaxf(acc[c][2], 0.f), fmaxf(acc[c][3], 0.f));
                float *dst = orow + (size_t)(co0 + c) * LP + p0;
                if (p0 + 3 < LP) *(float4 *)dst = v;  // LP is a multiple of 4 and >= L1: the padding lanes are never read
                else {
                    if (p0 < LP) dst[0] = v.x;
                    if (p0 + 1 < LP) dst[1] = v.y;
                    if (p0 + 2 < LP) dst[2] = v.z;
                }
            }
        }
    }
}

__host__ __device__ inline size_t cnn_conv_smem_bytes() {
    return (size_t)(CNN_C * CNN_K * CNN_C + CNN_C * CNN_TILE_IN + 3 * (CNN_TILE + 6) + 8 + CNN_C * CNN_K + CNN_C) * 4;
}

// ---- ConvTranspose1d(64 -> 2, k = 7, stride 3, pad 3) ---------------------------------------------------------------------
// out[co][j] = b[co] + sum_ci sum_{k = j%3 (+3, +6)} in[ci][(j + 3 - k) / 3] * w[ci][co][k]
// One thread per input position u produces the three outputs j = 3u, 3u+1, 3u+2 of both channels from in[ci][u-1],
// in[ci][u], in[ci][u+1]:  out[3u] = x[u+1] w0 + x[u] w3 + x[u-1] w6,  out[3u+1] = x[u+1] w1 + x[u] w4,
// out[3u+2] = x[u+1] w2 + x[u] w5  (three coalesced loads and 14 FMAs per input channel; the per-output summation
// order -- channels ascending, taps ascending -- is unchanged).
#define CNN_CONVT_THREADS 192  // 3 CTAs cover the 550 positions of an RNA004 read with 4 % idle threads
// `only` (optional): just the reads flagged there (tensor-core path: reads recomputed on the FP32 pipe).
__global__ void __launch_bounds__(CNN_CONVT_THREADS) cnn_convT_kernel(const float *act, const float *w4, const float *b4, int L1, int LP,
                                                        int Lout, float *scores, const int *only) {
    if (only && (only[-1] == 0 || only[blockIdx.y] == 0)) return;
    __shared__ __align__(16) float ws[CNN_C * 16];  // per ci: co0 k0..6, pad, co1 k0..6, pad
    for (int i = threadIdx.x; i < CNN_C * 16; i += blockDim.x) {
        const int ci = i >> 4, e = i & 15, co = e >> 3, k = e & 7;
        ws[i] = (k < CNN_K) ? w4[(ci * 2 + co) * CNN_K + k] : 0.0f;
    }
    __syncthreads();
    const int r = blockIdx.y;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (3 * u >= Lout) return;
    const float *ar = act + (size_t)r * CNN_C * LP;
    const float bias0 = b4[0], bias1 = b4[1];
    float o[2][3] = {{bias0, bias0, bias0}, {bias1, bias1, bias1}};
    const bool has_m = (u - 1 >= 0) && (u - 1 < L1), has_c = u < L1, has_p = u + 1 < L1;
#pragma unroll 8
    for (int ci = 0; ci < CNN_C; ci++) {
        const float *ap = ar + (size_t)ci * LP;
        const float xm = has_m ? ap[u - 1] : 0.0f, xc = has_c ? ap[u] : 0.0f, xp = has_p ? ap[u + 1] : 0.0f;
        const float4 wa = *reinterpret_cast<const float4 *>(ws + ci * 16), wb = *reinterpret_cast<const float4 *>(ws + ci * 16 + 4);
        const float4 wc = *reinterpret_cast<const float4 *>(ws + ci * 16 + 8), wd = *reinterpret_cast<const float4 *>(ws + ci * 16 + 12);
        // taps in ascending k: k = j%3 pairs with x[u+1], k+3 with x[u], k+6 with x[u-1]
        if (has_p) { o[0][0] = fmaf(xp, wa.x, o[0][0]); o[1][0] = fmaf(xp, wc.x, o[1][0]); }
        if (has_c) { o[0][0] = fmaf(xc, wa.w, o[0][0]); o[1][0] = fmaf(xc, wc.w, o[1][0]); }
        if (has_m) { o[0][0] = fmaf(xm, wb.z, o[0][0]); o[1][0] = fmaf(xm, wd.z, o[1][0]); }
        if (has_p) { o[0][1] = fmaf(xp, wa.y, o[0][1]); o[1][1] = fmaf(xp, wc.y, o[1][1]); }
        if (has_c) { o[0][1] = fmaf(xc, wb.x, o[0][1]); o[1][1] = fmaf(xc, wd.x, o[1][1]); }
        if (has_p) { o[0][2] = fmaf(xp, wa.z, o[0][2]); o[1][2] = fmaf(xp, wc.z, o[1][2]); }
        if (has_c) { o[0][2] = fmaf(xc, wb.y, o[0][2]); o[1][2] = fmaf(xc, wd.y, o[1][2]); }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const int j = 3 * u + c;
        if (j < Lout) {
            scores[((size_t)r * 2 + 0) * Lout + j] = o[0][c];
            scores[((size_t)r * 2 + 1) * Lout + j] = o[1][c];
        }
    }
}

// ---- post-processing (cnn.py:117-160) ---------------------------------------------------------------------------------
// argmax with numpy semantics: first maximum; a NaN wins over everything (first NaN)
__device__ __forceinline__ bool np_better(float v, int i, float bv, int bi) {
    const bool vn = !(v == v), bn = !(bv == bv);
    if (vn != bn) return vn;
    if (vn) return i < bi;
    return v > bv || (v == bv && i < bi);
}

__device__ int cta_argmax(const float *p, int n, float *sv, int *si) {
    float bv = -CUDART_INF_F;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = p[i];
        if (bi == 0x7fffffff || np_better(v, i, bv, bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(ADB_FULL, bv, o);
        const int oi = __shfl_xor_sync(ADB_FULL, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || np_better(ov, oi, bv, bi))) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
    __syncthreads();
    bv = sv[0]; bi = si[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++)
        if (si[w] != 0x7fffffff && (bi == 0x7fffffff || np_better(sv[w], si[w], bv, bi))) { bv = sv[w]; bi = si[w]; }
    __syncthreads();
    return bi == 0x7fffffff ? 0 : bi;
}

// one CTA (256 threads) per read: adapter argmax, mask, poly(A) argmax, mask (in place in scores[:, 1, :])
__global__ void __launch_bounds__(256) cnn_mask_kernel(float *scores, int Lout, int n_adapter_bins, int k, int *apos,
                                                       int *ppos) {
    __shared__ float sv[8];
    __shared__ int si[8];
    const int r = blockIdx.x;
    float *c0 = scores + ((size_t)r * 2) * Lout, *c1 = c0 + Lout;
    const int a = cta_argmax(c0, min(n_adapter_bins, Lout), sv, si);
    int p = 0;
    if (k >= 1) {
        for (int j = threadIdx.x; j < a; j += blockDim.x) c1[j] = CNN_SCORE_EXCL;
        __syncthreads();
        p = cta_argmax(c1, Lout, sv, si);
        if (k > 1)
            for (int j = p + 1 + threadIdx.x; j < Lout; j += blockDim.x) c1[j] = CNN_SCORE_EXCL;
    }
    if (threadIdx.x == 0) { apos[r] = a; ppos[r] = p; }
}

// flattened view of the poly(A) channel of one minibatch: element g of the flattened array = row g / Lout
struct FlatView {
    const float *scores;
    int Lout;
    int r0, nr;  // minibatch rows [r0, r0 + nr)
    __device__ __forceinline__ float at(long long g) const {
        const int rr = (int)(g / Lout), j = (int)(g % Lout);
        return scores[((size_t)(r0 + rr) * 2 + 1) * Lout + j];
    }
    __device__ __forceinline__ long long size() const { return (long long)nr * Lout; }
};

// Capacity of one row's peak list.  A local maximum's left edge i needs x[i-1] < x[i] and its plateau ends at
// ia > i with x[ia] < x[i]; no left edge lies in (i, ia], so consecutive left edges are at least two apart and a row
// of Lout scores lists at most ceil(Lout / 2) peaks.
__host__ __device__ inline int cnn_peak_cap(int Lout) { return Lout / 2 + 8; }

// pass A/B: local maxima (scipy _local_maxima_1d on the flattened minibatch array) whose LEFT EDGE lies in this row;
// midpoints are flattened indices and may fall into a later row when a plateau crosses row boundaries.
// One CTA (128 threads) per read.  pk_pos[r][pk_cap] (flattened midpoint), pk_cnt[r]; pk_cap = cnn_peak_cap(Lout).
__global__ void __launch_bounds__(128) cnn_peaks_kernel(const float *scores, int Lout, int batch_size, int n_reads,
                                                        int pk_cap, long long *pk_pos, int *pk_cnt) {
    __shared__ int wcount[4];
    __shared__ int base_sh;
    const int r = blockIdx.x;
    const int mb = r / batch_size;
    FlatView V{scores, Lout, mb * batch_size, min(batch_size, n_reads - mb * batch_size)};
    const long long N = V.size();
    const long long g0 = (long long)(r - V.r0) * Lout;
    const float *rowp = scores + ((size_t)r * 2 + 1) * Lout;  // the poly(A) channel of this read
    if (threadIdx.x == 0) base_sh = 0;
    __syncthreads();
    for (int jb = 0; jb < Lout; jb += blockDim.x) {
        const int j = jb + threadIdx.x;
        long long mid = -1;
        if (j < Lout) {
            const long long i = g0 + j;
            if (i >= 1 && i < N - 1) {
                // elements of this row straight from its pointer; only the neighbours across a row end go through the
                // flattened view (a 64-bit division per element)
                auto val = [&](long long g) { const long long jj = g - g0; return (jj >= 0 && jj < Lout) ? rowp[jj] : V.at(g); };
                const float xi = rowp[j];
                if (val(i - 1) < xi) {
                    long long ia = i + 1;
                    while (ia < N - 1 && val(ia) == xi) ia++;
                    if (val(ia) < xi) mid = (i + ia - 1) / 2;
                }
            }
        }
        const unsigned m = __ballot_sync(ADB_FULL, mid >= 0);
        if ((threadIdx.x & 31) == 0) wcount[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int off = base_sh;
        for (int w = 0; w < (int)(threadIdx.x >> 5); w++) off += wcount[w];
        if (mid >= 0) {
            const int pos = off + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
            pk_pos[(size_t)r * pk_cap + pos] = mid;
        }
        __syncthreads();
        if (threadIdx.x == 0) base_sh += wcount[0] + wcount[1] + wcount[2] + wcount[3];
        __syncthreads();
    }
    if (threadIdx.x == 0) pk_cnt[r] = base_sh;
}

// distance filter + per-read top-k.  One CTA (128 threads) per read: gathers the peaks listed under rows r-1, r, r+1 of
// the same minibatch (a distance-5 chain across a row boundary needs unmasked scores on both sides of it; chains
// spanning more than the neighbouring row do not occur), orders them by priority, runs scipy's greedy
// _select_by_peak_distance, keeps the survivors whose midpoint lies in row r, sorts those by (-height, position)
// and writes the first k positions (row-local).  cand[r][k] (0-padded), ncand[r].
// The working set holds up to three lists of pk_cap peaks: ws_cap = cnn_topk_ws_cap(pk_cap) entries of position,
// height, compaction slot and state (CNN_WS_BYTES_PER_PEAK bytes each).  It lives in dynamic shared memory
// (ws_glob == nullptr, one CTA per read) or, for windows whose working set does not fit there, in a slice of
// ws_glob per CTA, the CTAs then striding over the reads.
#define CNN_WS_BYTES_PER_PEAK 15
__host__ __device__ inline int cnn_topk_ws_cap(int pk_cap) { return (3 * pk_cap + 15) & ~15; }
__host__ __device__ inline size_t cnn_topk_ws_bytes(int ws_cap) { return (size_t)ws_cap * CNN_WS_BYTES_PER_PEAK; }
__global__ void __launch_bounds__(128) cnn_topk_kernel(const float *scores, int Lout, int batch_size, int n_reads, int k,
                                                       int dist, int pk_cap, int ws_cap, unsigned char *ws_glob,
                                                       const long long *pk_pos, const int *pk_cnt, int *cand, int *ncand) {
    extern __shared__ __align__(16) unsigned char ws_smem[];
    unsigned char *ws = ws_glob ? ws_glob + cnn_topk_ws_bytes(ws_cap) * blockIdx.x : ws_smem;
    long long *pos = (long long *)ws;                                   // flattened positions, ascending
    float *hgt = (float *)(pos + ws_cap);
    unsigned short *ord = (unsigned short *)(hgt + ws_cap);             // survivors of this row (compaction scratch)
    unsigned char *keep = (unsigned char *)(ord + ws_cap);              // 2 undecided, 1 kept, 0 removed
    __shared__ int n_sh;
    __shared__ int take_sh[2];
    for (int r = blockIdx.x; r < n_reads; r += gridDim.x) {
        __syncthreads();  // the previous read's working set is consumed
        const int mb = r / batch_size;
        FlatView V{scores, Lout, mb * batch_size, min(batch_size, n_reads - mb * batch_size)};
        const int rl = r - V.r0;
        // gather: the peaks of this row plus those of the neighbouring rows that can interact with them.  The distance
        // suppression only propagates through consecutive peaks closer than `dist`, so from either end of the row the
        // neighbour's list is followed only while its gaps stay below `dist` (usually not a single peak: the head of every
        // row is the masked stretch in front of the adapter end).  Lists are ascending and rows consecutive, so the
        // concatenation is ascending.  Each part is at most one list: n <= 3 * pk_cap <= ws_cap.
        const int c_mid = pk_cnt[r];
        const long long lo = (long long)rl * Lout, hi = lo + Lout;
        if (threadIdx.x == 0) {
            int tl = 0, tr = 0;
            const long long *pm = pk_pos + (size_t)r * pk_cap;
            long long first_pos = (c_mid > 0) ? pm[0] : 0x7fffffffffffffffLL, last_pos = (c_mid > 0) ? pm[c_mid - 1] : -1;
            if (rl > 0) {
                // trailing peaks of the previous row's list: a plateau that starts there can have its midpoint in this row
                // (always taken); further back only while the gaps stay below dist
                const long long *pl = pk_pos + (size_t)(r - 1) * pk_cap;
                const int cl = pk_cnt[r - 1];
                long long nxt = first_pos;
                while (tl < cl) {
                    const long long p = pl[cl - 1 - tl];
                    if (!(p >= lo || (dist > 0 && nxt != 0x7fffffffffffffffLL && nxt - p < dist))) break;
                    nxt = p; tl++;
                    if (last_pos < 0) last_pos = p;
                }
            }
            if (rl + 1 < V.nr && dist > 0 && last_pos >= 0) {
                const long long *pr = pk_pos + (size_t)(r + 1) * pk_cap;
                const int cr = pk_cnt[r + 1];
                long long prv = last_pos;
                while (tr < cr && pr[tr] - prv < dist) { prv = pr[tr]; tr++; }
            }
            take_sh[0] = tl; take_sh[1] = tr;
        }
        __syncthreads();
        int n = 0;
        for (int part = 0; part < 3; part++) {
            const int rr = r - 1 + part;
            int c, first;
            if (part == 0) { c = take_sh[0]; first = (c > 0) ? pk_cnt[r - 1] - c : 0; }
            else if (part == 1) { c = c_mid; first = 0; }
            else { c = take_sh[1]; first = 0; }
            for (int i = threadIdx.x; i < c; i += blockDim.x) {
                const long long p = pk_pos[(size_t)rr * pk_cap + first + i];
                pos[n + i] = p;
                hgt[n + i] = V.at(p);
                keep[n + i] = 2;
            }
            n += c;
        }
        // priority order (np.argsort of the heights, stable: ties keep the lower index first; scipy walks it from the back):
        // peak t has priority over peak i iff (height, index) of t is the larger pair.  Only peaks closer than `dist` are
        // ever compared, so no sorted order is materialised.
        auto over = [&](int t, int i) { const float ht = hgt[t], hi_ = hgt[i]; return (ht > hi_) || (ht == hi_ && t > i); };
        __syncthreads();
        // _select_by_peak_distance: in priority order a kept peak removes everything closer than `dist`; equivalently a peak
        // is kept iff no KEPT peak of higher priority lies within the distance.  Resolved in parallel rounds: a peak
        // decides once all its higher-priority neighbours have decided (the highest of every neighbourhood at once).
        // A round reads the states in bits 0-1 and writes the new state of its own peaks into bits 2-3 (a peak's byte has
        // one writer; readers mask), which become the state after the barrier.
        if (dist > 0) {
            bool pending = true;
            while (__syncthreads_or(pending)) {
                pending = false;
                for (int i = threadIdx.x; i < n; i += blockDim.x) {
                    unsigned char st = keep[i] & 3;
                    if (st == 2) {
                        bool killed = false, wait = false;
                        for (int t = i - 1; t >= 0 && pos[i] - pos[t] < dist; t--)
                            if (over(t, i)) { const unsigned char s2 = keep[t] & 3; killed |= (s2 == 1); wait |= (s2 == 2); }
                        for (int t = i + 1; t < n && pos[t] - pos[i] < dist; t++)
                            if (over(t, i)) { const unsigned char s2 = keep[t] & 3; killed |= (s2 == 1); wait |= (s2 == 2); }
                        if (killed) st = 0;
                        else if (!wait) st = 1;
                        else pending = true;
                    }
                    keep[i] = (unsigned char)((keep[i] & 3) | (st << 2));
                }
                __syncthreads();
                for (int i = threadIdx.x; i < n; i += blockDim.x) keep[i] = keep[i] >> 2;
            }
        } else {
            for (int i = threadIdx.x; i < n; i += blockDim.x) keep[i] = 1;
        }
        __syncthreads();
        // survivors in row r, best first: (-height, position); compacted, then ranked by counting among themselves
        if (threadIdx.x == 0) n_sh = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            if (keep[i] == 1 && pos[i] >= lo && pos[i] < hi) ord[atomicAdd(&n_sh, 1)] = (unsigned short)i;
        __syncthreads();
        const int ns = n_sh;
        for (int a = threadIdx.x; a < ns; a += blockDim.x) {
            const int i = ord[a];
            const float h = hgt[i];
            int rank = 0;
            for (int b = 0; b < ns; b++) {
                const int j = ord[b];
                const float hj = hgt[j];
                rank += (hj > h) || (hj == h && j < i);
            }
            if (rank < k) cand[(size_t)r * k + rank] = (int)(pos[i] - lo);
        }
        if (threadIdx.x == 0) ncand[r] = ns;
    }
}

// groups of candidates are assigned to rows in order of appearance (cnn.py:149-158): read r's candidates land in row
// (number of earlier reads of the minibatch that have at least one candidate).  One CTA per minibatch.
__global__ void __launch_bounds__(256) cnn_shift_kernel(const int *apos, const int *ppos, const int *cand, const int *ncand,
                                                        int batch_size, int n_reads, int k, int ds, int A0, int *given) {
    __shared__ int wtot[8];
    __shared__ int carry;
    const int mb = blockIdx.x;
    const int r0 = mb * batch_size, nr = min(batch_size, n_reads - r0);
    const int stride = 1 + max(k, 1);
    if (threadIdx.x == 0) carry = 0;
    // adapter ends + zero-filled candidate rows
    for (int i = threadIdx.x; i < nr; i += blockDim.x) {
        int *g = given + (size_t)(r0 + i) * stride;
        const int a = apos[r0 + i];
        g[0] = (a == 0) ? 0 : a * ds + A0;  // preds == min_obs_adapter -> 0 (cnn.py:179)
        for (int t = 0; t < max(k, 1); t++) g[1 + t] = 0;
        if (k == 1) { const int p = ppos[r0 + i]; g[1] = (p == 0) ? 0 : p * ds + A0; }
    }
    __syncthreads();
    if (k <= 1) return;
    for (int base = 0; base < nr; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int has = (i < nr && ncand[r0 + i] > 0) ? 1 : 0;
        const unsigned m = __ballot_sync(ADB_FULL, has);
        if ((threadIdx.x & 31) == 0) wtot[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int off = carry;
        for (int w = 0; w < (int)(threadIdx.x >> 5); w++) off += wtot[w];
        if (has) {
            const int row = off + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
            int *g = given + (size_t)(r0 + row) * stride;
            const int nc = min(ncand[r0 + i], k);
            for (int t = 0; t < nc; t++) {
                const int p = cand[(size_t)(r0 + i) * k + t];
                g[1 + t] = (p == 0) ? 0 : p * ds + A0;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) { int s = 0; for (int w = 0; w < 8; w++) s += wtot[w]; carry += s; }
        __syncthreads();
    }
}

// ---- host orchestration -----------------------------------------------------------------------------------------------------
struct CnnDims {
    int Lx, L1, LP, Lout;
};
static CnnDims cnn_dims(int m, int A0, int f) {
    CnnDims d;
    d.Lx = (std::max(m - A0, 0) + f - 1) / f;
    d.L1 = (d.Lx + 2 * 3 - CNN_K) / 3 + 1;
    d.LP = (d.L1 + 3) & ~3;
    d.Lout = (d.L1 - 1) * 3 - 2 * 3 + CNN_K;
    return d;
}

// x [n][Lx] (device) -> scores [n][2][Lout] (device); chunked over reads to bound the activation buffers
// tensor-core version of the two 64 -> 64 convolutions (adb_cnn_tc.cuh)
__global__ void cnn_tc_pack_weights_kernel(const float *w, __half *packed);
static int cnn_tc_launch_setup();
// Layer 3's epilogue multiplies every activation with the 14 weights of the transposed convolution.  From shared memory
// that is two 16-byte broadcast loads per channel and thread -- 512 B of register-file writes per warp and load, the
// bottleneck of the epilogue.  From the CONSTANT bank the weights reach the FFMAs through the uniform datapath (ULDC +
// uniform-register operands): no vector register is written.  One slot per context ([co][ci][8] weights + the 64 layer-3
// biases), filled stream-ordered by a device-to-device copy into the symbol (cnn_ct_pack_kernel -> cudaMemcpyToSymbolAsync).
#define ADB_CT_SLOTS 4
#define ADB_CT_FLOATS (2 * 64 * 8 + 64)
__constant__ float adb_c_convT[ADB_CT_SLOTS][ADB_CT_FLOATS];

__global__ void cnn_ct_pack_kernel(const float *w4 /* torch layout [ci][co][k] */, const float *b3, float *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 1024) {
        const int co = i >> 9, ci = (i >> 3) & 63, k = i & 7;
        out[i] = (k < CNN_K) ? w4[(ci * 2 + co) * CNN_K + k] : 0.0f;
    } else if (i < ADB_CT_FLOATS) {
        out[i] = b3[i - 1024];
    }
}

static void cnn_tc_launch(int layer, const void *in, void *out, const __half *wp, const float *bias, const float *w1,
                          const float *b1, int n_reads, int Lx, int L1, int LP, int *redo, int sm_count, cudaStream_t st, int cslot = -1);
static size_t cnn_tc_a0t_bytes_per_read(int L1);
static int cnn_tc_a0t_rows_host(int L1);

static int cnn_forward_dev(adb_ctx *ctx, const float *x, int n, const CnnDims &D, const float *w_dev, float *scores,
                           cudaStream_t st) {
    if (ctx->cnn_w.ensure(sizeof(float) * 2 * CNN_C * CNN_K * CNN_C)) { set_err("cudaMalloc cnn weights"); return ADB_ERR_CUDA; }
    float *packed = (float *)ctx->cnn_w.p;
    {
        KernelTimer t(ctx, 6, st);
        cnn_pack_weights_kernel<<<(2 * CNN_C * CNN_K * CNN_C + 255) / 256, 256, 0, st>>>(w_dev, packed);
    }
    ctx->launches += 1;
    const size_t act_per_read = (size_t)CNN_C * D.LP * sizeof(float);
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)1 << 30) / act_per_read));
    if (ctx->cnn_act0.ensure(act_per_read * chunk) || ctx->cnn_act1.ensure(act_per_read * chunk)) {
        set_err("cudaMalloc cnn activations");
        return ADB_ERR_CUDA;
    }
    const size_t smem = cnn_conv_smem_bytes();
    CUDA_TRY(cudaFuncSetAttribute(cnn_conv64_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaFuncSetAttribute(cnn_conv64_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    float *a0 = (float *)ctx->cnn_act0.p, *a1 = (float *)ctx->cnn_act1.p;
    const bool use_tc = !ctx->opt_cnn_fp32;
    __half *wtc = nullptr;
    unsigned char *a0t = nullptr;
    int *redo = nullptr;
    int cslot = -1;  // slot of the constant bank holding the transposed convolution's weights (-1: shared memory)
    if (use_tc) {
        // split fp16 weights of both layers, then the per-read "outside the fp16 range" flags of one chunk
        const size_t wbytes = sizeof(__half) * 2 * CNN_K * 2 * 4096;
        if (ctx->cnn_wtc.ensure(wbytes + sizeof(int) * ((size_t)chunk + 4))) { set_err("cudaMalloc cnn tc weights"); return ADB_ERR_CUDA; }
        wtc = (__half *)ctx->cnn_wtc.p;
        redo = (int *)((unsigned char *)ctx->cnn_wtc.p + wbytes) + 4;  // redo[-1] = "any read of the chunk flagged"
        {
            KernelTimer t(ctx, 6, st);
            cnn_tc_pack_weights_kernel<<<(2 * CNN_K * 4096 + 255) / 256, 256, 0, st>>>(w_dev, wtc);
        }
        ctx->launches += 1;
        if (ctx->ct_slot >= 0 && !getenv("ADB_NO_CONST_CONVT")) {
            // the transposed convolution's weights + layer 3's biases into this context's slot of the constant bank
            if (ctx->cnn_ct.ensure(sizeof(float) * ADB_CT_FLOATS)) { set_err("cudaMalloc cnn constants"); return ADB_ERR_CUDA; }
            cnn_ct_pack_kernel<<<(ADB_CT_FLOATS + 255) / 256, 256, 0, st>>>(w_dev + CNN_W4, w_dev + CNN_B3, (float *)ctx->cnn_ct.p);
            CUDA_TRY(cudaMemcpyToSymbolAsync(adb_c_convT, ctx->cnn_ct.p, sizeof(float) * ADB_CT_FLOATS,
                                             sizeof(float) * ADB_CT_FLOATS * (size_t)ctx->ct_slot, cudaMemcpyDeviceToDevice, st));
            ctx->launches += 1;
            cslot = ctx->ct_slot;
        }
        if (cnn_tc_launch_setup()) { set_err("cudaFuncSetAttribute cnn tc"); return ADB_ERR_CUDA; }
        // layer 2 -> layer 3 activations in layer 3's tile layout; the padding rows are never written: zero them whenever
        // the buffer is (re)allocated
        const size_t a0t_bytes = cnn_tc_a0t_bytes_per_read(D.L1) * (size_t)chunk;
        const void *before = ctx->cnn_a0t.p;
        const size_t cap_before = ctx->cnn_a0t.cap;
        if (ctx->cnn_a0t.ensure(a0t_bytes)) { set_err("cudaMalloc cnn a0t"); return ADB_ERR_CUDA; }
        // (also when L1 changes: rows between the old and the new end would keep activations of the old geometry)
        if (ctx->cnn_a0t.p != before || ctx->cnn_a0t.cap != cap_before || ctx->cnn_a0t_l1 != D.L1)
            CUDA_TRY(cudaMemsetAsync(ctx->cnn_a0t.p, 0, ctx->cnn_a0t.cap, st));
        ctx->cnn_a0t_l1 = D.L1;
        a0t = (unsigned char *)ctx->cnn_a0t.p;
    }
    for (int r0 = 0; r0 < n; r0 += chunk) {
        const int nc = std::min(chunk, n - r0);
        const int tiles = nc * ((D.L1 + CNN_TILE - 1) / CNN_TILE);
        const int grid = std::max(1, std::min(tiles, ctx->sm_count));
        if (use_tc) {
            CUDA_TRY(cudaMemsetAsync(redo - 4, 0, sizeof(int) * ((size_t)nc + 4), st));
            {
                KernelTimer t(ctx, 5, st);
                cnn_tc_launch(2, x + (size_t)r0 * D.Lx, a0t, wtc, w_dev + CNN_B2, w_dev + CNN_W1, w_dev + CNN_B1, nc, D.Lx, D.L1,
                              cnn_tc_a0t_rows_host(D.L1), redo, ctx->sm_count, st);
            }
            {
                KernelTimer t(ctx, 5, st);
                // layer 3 + the transposed convolution: scores straight from the epilogue
                cnn_tc_launch(3, a0t, scores + (size_t)r0 * 2 * D.Lout, wtc + (size_t)CNN_K * 2 * 4096, w_dev + CNN_B3,
                              w_dev + CNN_W4, w_dev + CNN_B4, nc, D.Lout, D.L1, cnn_tc_a0t_rows_host(D.L1), redo,
                              ctx->sm_count, st, cslot);
            }
            {
                // reads with a value outside the fp16 range (flagged by either layer): both layers again on the FP32 pipe
                KernelTimer t(ctx, 7, st);
                cnn_conv64_kernel<true><<<grid, CNN_THREADS, smem, st>>>(x + (size_t)r0 * D.Lx, a0, packed, w_dev + CNN_B2,
                                                                          w_dev + CNN_W1, w_dev + CNN_B1, nc, D.Lx, D.L1, D.LP, redo);
                cnn_conv64_kernel<false><<<grid, CNN_THREADS, smem, st>>>(a0, a1, packed + CNN_C * CNN_K * CNN_C, w_dev + CNN_B3,
                                                                           nullptr, nullptr, nc, D.Lx, D.L1, D.LP, redo);
            }
            ctx->launches += 2;
        } else {
        {
            KernelTimer t(ctx, 5, st);
            cnn_conv64_kernel<true><<<grid, CNN_THREADS, smem, st>>>(x + (size_t)r0 * D.Lx, a0, packed, w_dev + CNN_B2,
                                                                      w_dev + CNN_W1, w_dev + CNN_B1, nc, D.Lx, D.L1, D.LP, nullptr);
        }
        {
            KernelTimer t(ctx, 5, st);
            cnn_conv64_kernel<false><<<grid, CNN_THREADS, smem, st>>>(a0, a1, packed + CNN_C * CNN_K * CNN_C, w_dev + CNN_B3,
                                                                       nullptr, nullptr, nc, D.Lx, D.L1, D.LP, nullptr);
        }
        }
        {
            // FP32 path: every read; tensor-core path: only the reads redone on the FP32 pipe (the others got their
            // scores from layer 3's epilogue)
            KernelTimer t(ctx, use_tc ? 7 : 5, st);
            dim3 g(((D.Lout + 2) / 3 + CNN_CONVT_THREADS - 1) / CNN_CONVT_THREADS, nc);
            cnn_convT_kernel<<<g, CNN_CONVT_THREADS, 0, st>>>(a1, w_dev + CNN_W4, w_dev + CNN_B4, D.L1, D.LP, D.Lout,
                                                scores + (size_t)r0 * 2 * D.Lout, use_tc ? redo : nullptr);
        }
        ctx->launches += 3;
    }
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

// primary boundaries of the CNN method -> given[n_reads][1 + max(k,1)]
static int cnn_primary_boundaries(adb_ctx *ctx, const BatchDev &B, const adb_config &cfg, const float *w_dev, int *given,
                                  cudaStream_t st) {
    const CnnDims D = cnn_dims(B.m, cfg.min_obs_adapter, cfg.downscale_factor);
    if (D.Lx < CNN_K || D.Lout < 3) {
        set_err("preload window outside the range supported by the CNN kernels");
        return ADB_ERR_UNSUPPORTED;
    }
    const int pk_cap = cnn_peak_cap(D.Lout), ws_cap = cnn_topk_ws_cap(pk_cap);
    if (ws_cap > 65536) {
        // cnn_topk_kernel compacts the survivors by 16-bit working-set index (windows up to about 437 000 samples at
        // downscale factor 10)
        set_err("preload window too long for the 16-bit working-set indices of cnn_topk_kernel");
        return ADB_ERR_UNSUPPORTED;
    }
    const int n = B.n_reads, k = cfg.polya_cand_k;
    if (ctx->cnn_x.ensure(sizeof(float) * (size_t)n * D.Lx) || ctx->cnn_scores.ensure(sizeof(float) * (size_t)n * 2 * D.Lout)) {
        set_err("cudaMalloc cnn buffers");
        return ADB_ERR_CUDA;
    }
    float *x = (float *)ctx->cnn_x.p, *scores = (float *)ctx->cnn_scores.p;
    {
        const size_t smem = (((size_t)D.Lx * 4 + 15) & ~(size_t)15) + ((ADB_SEL_SMEM_BYTES + 15) & ~15) + 64;
        CUDA_TRY(cudaFuncSetAttribute(cnn_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        KernelTimer t(ctx, 6, st);
        const size_t wsm = cnn_prep_warp_smem(D.Lx);
        if (B.sig_type == ADB_SIG_I16 && (int)wsm <= ctx->max_smem_optin && !getenv("ADB_PREP_CTA") &&
            (((D.Lx + 3) & ~3) * 4 - 16) / (2 * cfg.downscale_factor) >= 32) {
            CUDA_TRY(cudaFuncSetAttribute(cnn_prep_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm));
            int occ = 0;
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cnn_prep_warp_kernel, PREP_WARPS * 32, wsm));
            const int grid = std::max(1, std::min((n + PREP_WARPS - 1) / PREP_WARPS, ctx->sm_count * std::max(occ, 1)));
            cnn_prep_warp_kernel<<<grid, PREP_WARPS * 32, wsm, st>>>(B, cfg.min_obs_adapter, cfg.downscale_factor, D.Lx, x);
        } else {
            cnn_prep_kernel<<<n, 256, smem, st>>>(B, cfg.min_obs_adapter, cfg.downscale_factor, D.Lx, x);
        }
        ctx->launches += 1;
    }
    int rc = cnn_forward_dev(ctx, x, n, D, w_dev, scores, st);
    if (rc) return rc;
    // cnn_topk_kernel's working set: dynamic shared memory (one CTA per read) where it fits, else a slice of global
    // scratch per CTA of a grid striding over the reads
    const size_t ws_bytes = cnn_topk_ws_bytes(ws_cap);
    const bool ws_in_smem = (int)(ws_bytes + 64) <= ctx->max_smem_optin;
    const int topk_grid = ws_in_smem ? n : std::max(1, std::min(n, ctx->sm_count * 8));
    // post-processing scratch: pk_pos [n][pk_cap] int64; apos, ppos, pk_cnt, ncand [n] ints; cand [n][k];
    // [topk_grid] working sets (global variant only)
    const size_t ints = (size_t)n * (4 + std::max(k, 1));
    const size_t ws_off = (sizeof(long long) * (size_t)n * pk_cap + sizeof(int) * ints + 15) & ~(size_t)15;
    if (ctx->cnn_post.ensure(ws_off + (ws_in_smem ? 0 : ws_bytes * (size_t)topk_grid) + 64)) {
        set_err("cudaMalloc cnn post-processing");
        return ADB_ERR_CUDA;
    }
    long long *pk_pos = (long long *)ctx->cnn_post.p;
    int *apos = (int *)(pk_pos + (size_t)n * pk_cap), *ppos = apos + n, *pk_cnt = ppos + n, *ncand = pk_cnt + n;
    int *cand = ncand + n;
    unsigned char *ws_glob = ws_in_smem ? nullptr : (unsigned char *)ctx->cnn_post.p + ws_off;
    const int nadp = (cfg.max_obs_adapter - cfg.min_obs_adapter) / cfg.downscale_factor;
    const int n_batches = (n + B.batch_size - 1) / B.batch_size;
    {
        KernelTimer t(ctx, 6, st);
        cnn_mask_kernel<<<n, 256, 0, st>>>(scores, D.Lout, nadp, k, apos, ppos);
    }
    ctx->launches += 1;
    if (k > 1) {
        CUDA_TRY(cudaMemsetAsync(cand, 0, sizeof(int) * (size_t)n * k, st));
        {
            KernelTimer t(ctx, 6, st);
            cnn_peaks_kernel<<<n, 128, 0, st>>>(scores, D.Lout, B.batch_size, n, pk_cap, pk_pos, pk_cnt);
        }
        {
            KernelTimer t(ctx, 6, st);
            const size_t sm = ws_in_smem ? ws_bytes : 0;
            if (ws_in_smem) CUDA_TRY(cudaFuncSetAttribute(cnn_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            cnn_topk_kernel<<<topk_grid, 128, sm, st>>>(scores, D.Lout, B.batch_size, n, k, 5, pk_cap, ws_cap, ws_glob,
                                                         pk_pos, pk_cnt, cand, ncand);
        }
        ctx->launches += 2;
    }
    {
        KernelTimer t(ctx, 6, st);
        cnn_shift_kernel<<<n_batches, 256, 0, st>>>(apos, ppos, cand, ncand, B.batch_size, n, k, cfg.downscale_factor,
                                                    cfg.min_obs_adapter, given);
    }
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}
