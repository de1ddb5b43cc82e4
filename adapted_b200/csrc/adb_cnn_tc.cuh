// Conv1d(64 -> 64, k = 7, pad 3) + ReLU of BoundariesCNN (adapted/detect/cnn.py:16-52, layers 2 and 3: 98 % of the
// 64.6 MFLOP per read) on the 5th-generation tensor cores: tcgen05.mma kind::f16, accumulators in TMEM.
//
// Implicit GEMM: out[t][co] = sum_k sum_ci in[ci][t + k - 3] * W[co][ci][k]  ->  for each of the 7 taps one
// [M = 128 positions][K = 64 ci] x [K][N = 64 co] product accumulated into the same TMEM tile.  The activation tile of
// a job (128 positions + 3 halo rows on each side) is kept in shared memory in the canonical K-major "interleaved"
// (no-swizzle) UMMA layout with the rows of consecutive 8-row groups contiguous:
//     element (position row q, channel ci)  at  ((ci / 8) * RA + q) * 16 B + (ci % 8) * 2 B
// so that tap k is simply the same tile with its start address advanced by k rows (k * 16 B) -- no im2col copy.
//
// Precision: the reference is float32 (torch CPU) and the boundary contract is +-1 downscaled step on arg-maxima of
// fairly flat score curves, which a single 11-bit operand does not keep.  Split arithmetic: every operand is
// x = hi + lo with hi = fp16(x) (11 significant bits) and lo = fp16(x - hi) (the next 11 bits; x - hi is exact in
// float32); the products hi*hi + lo*hi + hi*lo are exact in the tensor core and accumulate in float32 in TMEM (the
// dropped lo*lo term is 2^-22 relative) -- the same error budget as 3xTF32 at half the operand bytes and twice the
// MMA rate.  With 2-byte operands the split weights of a whole layer (7 taps x (hi, lo) x 8 KB = 112 KB) stay
// RESIDENT in shared memory for the CTA's life: nothing is streamed per tile.  Values outside the fp16 range
// (|x| >= 65504: pathological reads only) set a per-read flag; flagged reads are recomputed by the FP32-pipe kernel
// (cnn_conv64_kernel with a read filter), so the result never depends on the range.
//
// Pipeline (one persistent CTA per SM, warp-specialised, tiles double-buffered in shared memory and in TMEM):
//   issuer warp (one thread): waits for "tile buffer b built" and "accumulator b drained", issues the 84 MMAs of the
//                 tile and commits them to the accumulator barrier -- it runs ahead of the workers by up to one tile
//   8 worker warps, iteration i:
//                 (a) global loads of tile i+1 into registers            -- latency covered by (c)
//                 (c) epilogue of tile i-1: TMEM -> registers -> bias + ReLU -> global, accumulator handed back
//                 (d) split the prefetched registers into the hi / lo planes of the other tile buffer, hand it over
//   (mbarriers only; no CTA-wide barrier inside the loop)
// Layer 1 (1 -> 64, 0.8 % of the flops) is fused into (d) of layer 2 on the FP32 pipe, the transposed convolution
// (64 -> 2) stays in cnn_convT_kernel.
#pragma once
#include <cuda_fp16.h>

#include "adb_cnn.cuh"

#define TC_WORKERS 256                   // 8 worker warps
#define TC_THREADS (TC_WORKERS + 64)      // + the MMA issuer warp + the tile loader warp (layer 3)
#define TC_THREADS2 (2 * TC_WORKERS + 64)  // layer 2: 8 warps build the tiles, 8 more drain the accumulators, + issuer (+ idle loader)
#define TC_ROWS 128                      // output positions per job (one M = 128 tile)
#define TC_RA (TC_ROWS + 8)              // rows of the activation tile (6 halo rows, rounded to a multiple of 8)
#define TC_NQ (TC_ROWS + 6)              // rows actually filled
#define TC_PLANE (8 * TC_RA * 16)        // bytes of one activation plane (hi or lo): 8 channel octets x RA rows x 16 B
#define TC_WPART (8 * 64 * 16)           // bytes of one weight part of one tap: 8 channel octets x 64 co x 16 B
#define TC_WBYTES (CNN_K * 2 * TC_WPART) // resident weights of one layer: 114 688 B
#define TC_NX (3 * TC_NQ + 6)            // x samples under one tile of layer 1 (FUSE_L1)
#define TC_ITEMS (8 * TC_NQ)             // (octet, row) items of a tile: 8 channels each
#define TC_ROUNDS ((TC_ITEMS + TC_WORKERS - 1) / TC_WORKERS)
// instruction descriptor (cute/arch/mma_sm100_desc.hpp): D = f32 [4,6) = 1, A = B = f16 (0), both K-major,
// N >> 3 at [17,23), M >> 4 at [24,29)
#define TC_IDESC ((1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24))    // N = 64
#define TC_IDESC2 ((1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24))  // N = 128: [W_hi | W_lo] side by side

// weights: torch layout w[co][ci][k] -> [layer][tap][ci / 8][hi, lo][co][ci % 8] fp16: per tap and channel octet the 64
// rows of the hi part are followed by the 64 rows of the lo part, so that ONE N = 128 operand [W_hi | W_lo] serves the
// products hi * hi and hi * lo of an activation tile (the activation tile is read from shared memory once for both)
__global__ void cnn_tc_pack_weights_kernel(const float *w, __half *packed) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * CNN_K * 4096) return;
    const int layer = i / (CNN_K * 4096), rem = i % (CNN_K * 4096);
    const int k = rem / 4096, e = rem % 4096;
    const int kc = e / 512, co = (e / 8) % 64, j = e % 8;
    const int ci = kc * 8 + j;
    const float v = (w + (layer == 0 ? CNN_W2 : CNN_W3))[(co * CNN_C + ci) * CNN_K + k];
    const __half hi = __float2half_rn(v);
    __half *dst = packed + ((size_t)(layer * CNN_K + k) * 2) * 4096 + (size_t)kc * 1024 + co * 8 + j;
    dst[0] = hi;
    dst[512] = __float2half_rn(__fsub_rn(v, __half2float(hi)));
}

// SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), version 1
// [46,48), base offset 0, layout type SWIZZLE_NONE (0) [61,64).  Kept as two 32-bit halves: moving the start address
// is one 32-bit add on the low word (the tile never crosses the 14-bit field).
__device__ __forceinline__ uint32_t tc_desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
    return ((saddr >> 4) & 0x3fffu) | (((lbo_bytes >> 4) & 0x3fffu) << 16);
}
__device__ __forceinline__ uint32_t tc_desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3fffu) | (1u << 14); }

__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t accumulate, uint32_t idesc = TC_IDESC) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}

// one lane of a converged warp (elect.sync): ptxas then knows that a single thread issues the tcgen05 instructions and
// does not wrap each of them into a per-value serialisation loop
__device__ __forceinline__ bool tc_elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t v[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 8 channels of one row -> 16 B of the hi plane + 16 B of the lo plane; returns true if a value left the fp16 range
__device__ __forceinline__ bool tc_split_store(unsigned char *hi_plane, unsigned char *lo_plane, int kc, int q,
                                               const float v[8]) {
    __half2 h[4], l[4];
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const __half h0 = __float2half_rn(v[2 * j]), h1 = __float2half_rn(v[2 * j + 1]);
        const float f0 = __half2float(h0), f1 = __half2float(h1);
        bad |= !(fabsf(f0) <= 65504.0f) || !(fabsf(f1) <= 65504.0f);
        h[j] = __halves2half2(h0, h1);
        l[j] = __halves2half2(__float2half_rn(__fsub_rn(v[2 * j], f0)), __float2half_rn(__fsub_rn(v[2 * j + 1], f1)));
    }
    const size_t off = ((size_t)kc * TC_RA + q) * 16;
    *reinterpret_cast<uint4 *>(hi_plane + off) = *reinterpret_cast<const uint4 *>(h);
    *reinterpret_cast<uint4 *>(lo_plane + off) = *reinterpret_cast<const uint4 *>(l);
    return bad;
}

// Row stream of a chunk.  The reads of a chunk lie end to end, S rows apart: read r's position p is stream row
// g = r S + p.  With S = L1 + 3 ("packed", the default) the three rows behind every read are exactly the zero padding a
// k = 7, pad 3 convolution needs on both sides of a read, and the +-1-row neighbours of the fused transposed
// convolution are zero as well, so tiles walk the stream without regard to read boundaries:
//     layer 2: tile j covers rows 128 j ..;   layer 3: tile j covers rows 126 j - 1 .. (two rows overlap, see below)
// A row that is not a position of a read of the chunk (a gap row, a row in front of the stream or behind its last read)
// is zero padding.  Per-read tiling (option "cnn_tc_per_read_tiles", the previous scheme, kept as the A/B arm) is the
// same stream with S the per-read block below and the tiles restarting at every read.
//
// Intermediate activations between the two layers ("A0T"): layer 2's epilogue writes its output already split into the
// fp16 hi / lo planes and in the row order of layer 3's shared-memory tile,
//     A0T[plane][ci / 8][rho = g + TC_A0T_PAD][ci % 8]      (16 B per row, `a0t_rows` rows per octet),
// so that the operand tile of a layer-3 job is 16 contiguous runs of 134 rows: sixteen cp.async.bulk copies per tile,
// no thread touches the data.  Layer 2 writes every row its tiles cover, gap rows as zeros; the rows in front of the
// stream (and, with per-read tiling, the rows between a read's last tile and the next read) are never written and stay
// zero from the buffer's memset.
#define TC_A0T_PAD 4                                        // zero rows in front of the stream
#define TC_L3_STRIDE (TC_ROWS - 2)                          // layer 3 tiles overlap by two rows (fused convT, see below)
#define TC_GAP 3                                            // zero rows behind every read of the packed stream

struct TcTiles {
    int S;       // rows per read
    int stride;  // rows a tile advances: TC_ROWS (layer 2) or TC_L3_STRIDE (layer 3)
    int jpr;     // tiles per segment: per read (per-read tiling) or the whole chunk (packed)
    int n_jobs;
    // first row of tile `job` (layer 3: the row in front of its first output row, as seen from rho = g + TC_A0T_PAD)
    __host__ __device__ int row0(int job) const { return (job / jpr) * S + (job % jpr) * stride; }
};
__host__ __device__ inline int cnn_tc_read_rows(int L1, int per_read) {
    if (!per_read) return L1 + TC_GAP;
    // one block per read: what its layer 2 tiles write (rho up to 128 J2 + 3) and what its last layer 3 tile reads
    // (rho up to 126 (J3 - 1) + 133), whichever is larger
    const int j2 = (L1 + TC_ROWS - 1) / TC_ROWS, j3 = (L1 + TC_L3_STRIDE - 1) / TC_L3_STRIDE;
    const int w = TC_ROWS * j2 + TC_A0T_PAD, rd = TC_L3_STRIDE * (j3 - 1) + TC_NQ;
    return ((w > rd ? w : rd) + 7) & ~7;
}
__host__ __device__ inline TcTiles cnn_tc_tiles(int layer, int n_reads, int L1, int per_read) {
    TcTiles t;
    t.S = cnn_tc_read_rows(L1, per_read);
    t.stride = layer == 3 ? TC_L3_STRIDE : TC_ROWS;
    if (per_read) {
        t.jpr = (L1 + t.stride - 1) / t.stride;
        t.n_jobs = n_reads * t.jpr;
    } else {
        t.n_jobs = (int)(((long long)n_reads * t.S + t.stride - 1) / t.stride);
        t.jpr = t.n_jobs;
    }
    return t;
}
// rows per octet of A0T for chunks of up to n_reads reads: what layer 2's last tile writes and what layer 3's last tile
// reads, whichever is larger; the kernels get it in their `LP` argument
__host__ __device__ inline int cnn_tc_a0t_rows(int n_reads, int L1, int per_read) {
    const TcTiles t2 = cnn_tc_tiles(2, n_reads, L1, per_read), t3 = cnn_tc_tiles(3, n_reads, L1, per_read);
    const int w = t2.row0(t2.n_jobs - 1) + TC_ROWS + TC_A0T_PAD, rd = t3.row0(t3.n_jobs - 1) + TC_NQ;
    return ((w > rd ? w : rd) + 7) & ~7;
}
// stream row g -> (read, position); true if it is a position of a read of the chunk.  g >= -TC_A0T_PAD > -S: the rows in
// front of the stream give read 0 and a negative position.
__device__ __forceinline__ bool tc_row_read(int g, int S, int L1, int n_reads, int &r, int &p) {
    r = g / S;
    p = g - r * S;
    return (unsigned)p < (unsigned)L1 && r < n_reads;
}
#define TC_TILE_RUN (TC_NQ * 16)                            // bytes of one (plane, octet) run of a tile

__host__ __device__ inline size_t cnn_tc_smem_bytes_layer(int layer) {
    if (layer == 3)  // weights + 3 tile buffers + W4s [2][64][8] + edge sums + bias + barriers
        return (size_t)TC_WBYTES + 3 * 2 * (size_t)TC_PLANE + 1024 * 4 + 64 * 4 + 64 * 4 + 160 + 256;
    return (size_t)TC_WBYTES + 2 * 2 * (size_t)TC_PLANE + (size_t)(TC_NX + 10) * 4 + 64 * 8 * 4 + 64 * 4 + 160 + 1024;
}

// LAYER 2: in = x [N][Lx] with the row stride Lx = 3 S_packed samples (zeros behind each read's samples: stream row g
//   takes its layer-1 inputs from x[3 g - 3 .. 3 g + 3] across read boundaries), layer 1 fused into the operand build;
//   out = A0T.
// LAYER 3: in = A0T, out = scores [N][2][Lout]: the transposed convolution (64 -> 2, k = 7, stride 3, pad 3) is fused
//   into the epilogue, layer 3's activations never leave the SM.  out[co][3u + c] needs the activations of positions
//   u - 1, u, u + 1; tiles of 128 rows therefore advance by 126 rows (rows t0 .. t0 + 127 with t0 = 126 j - 1
//   produce the outputs of rows t0 + 1 .. t0 + 126) and nothing is exchanged between tiles.  Warp w (rows (w % 4) * 32 ..)
//   reads all 64 channels of its rows from TMEM and accumulates, for output channel co = w / 4, the seven per-tap
//   partial sums P_k = sum_ci act[ci][row] * W4[ci][co][k]; then out[3u] = P0(u+1) + P3(u) + P6(u-1),
//   out[3u+1] = P1(u+1) + P4(u), out[3u+2] = P2(u+1) + P5(u) with the neighbours' sums by shuffle (warp edges through
//   a 256-byte shared buffer, one named barrier per tile).  `w1` / `b1` carry W4 / b4, `Lx` carries Lout.
// wp  : packed weights of this layer, [7][2][4096] fp16 (cnn_tc_pack_weights_kernel)
// redo: [N] set to 1 for reads with a value outside the fp16 range (recomputed on the FP32 pipe afterwards)
// per_read: tiles restart at every read (cnn_tc_tiles)
template <int LAYER, int CSLOT = -1>  // CSLOT >= 0 (layer 3): transposed-convolution weights from that slot of adb_c_convT
__global__ void __launch_bounds__(LAYER == 2 ? TC_THREADS2 : TC_THREADS, 1) cnn_conv64_tc_kernel(const void *in, void *out, const __half *wp,
                                                                     const float *bias, const float *w1, const float *b1,
                                                                     int n_reads, int Lx, int L1, int LP, int per_read, int *redo) {
    constexpr int NBUF = LAYER == 3 ? 3 : 2;
    constexpr int NWW = LAYER == 2 ? 2 * TC_WORKERS / 32 : TC_WORKERS / 32;  // worker warps (layer 2: builders + drainers)
    const int a0t_rows = LP;                                    // rows per octet of A0T (cnn_tc_a0t_rows)
    const TcTiles T = cnn_tc_tiles(LAYER, n_reads, L1, per_read);
    extern __shared__ __align__(1024) unsigned char tsm[];
    unsigned char *Wsm = tsm;                                   // resident weights [7][hi, lo][8][64][8] fp16
    unsigned char *Abuf = tsm + TC_WBYTES;                      // NBUF tile buffers x (hi plane, lo plane)
    float *Xs = (float *)(Abuf + NBUF * 2 * TC_PLANE);          // LAYER 2: x window of the tile being built
    float *W1s = Xs + TC_NX + 10;                               // LAYER 2: [64][7] + [64]
    float *W4s = Xs;                                            // LAYER 3: [co][ci][8] (7 taps + pad) = 1024 floats
    float *Eg = W4s + 1024;                                     // LAYER 3: [2 tiles][2 co][4 warps][4] edge partial sums
    float *Bs = (LAYER == 3 ? Eg + 64 : W1s + 64 * 8);          // bias [64]
    // barriers: accb[2] accumulator complete (tcgen05.commit), afull[NBUF] tile buffer ready (layer 2: all workers,
    // layer 3: the bulk copies), accfree[2] accumulator drained by the epilogue (all workers)
    uint64_t *accb = (uint64_t *)(((uintptr_t)(Bs + 64) + 15) & ~(uintptr_t)15);
    uint64_t *afull = accb + 2, *accfree = accb + 2 + NBUF;
    uint64_t *sfree = accfree + 2;  // [NBUF] layer 3: the MMAs reading tile buffer b are complete (second commit)
    uint32_t *tmem_slot = (uint32_t *)(sfree + NBUF);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int b = 0; b < 2; b++) { mbar_init(&accb[b], 1); mbar_init(&accfree[b], TC_WORKERS); }
        for (int b = 0; b < NBUF; b++) { mbar_init(&afull[b], LAYER == 3 ? 1 : TC_WORKERS); mbar_init(&sfree[b], 1); }
    }
    for (int i = tid; i < TC_WBYTES / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(Wsm)[i] = reinterpret_cast<const uint4 *>(wp)[i];
    if (LAYER == 2) {
        for (int i = tid; i < CNN_C * CNN_K; i += blockDim.x) W1s[i] = w1[i];
        for (int i = tid; i < CNN_C; i += blockDim.x) W1s[CNN_C * CNN_K + i] = b1[i];
    } else {
        for (int i = tid; i < 1024; i += blockDim.x) {  // torch layout W4[ci][co][k]
            const int co = i >> 9, ci = (i >> 3) & 63, k = i & 7;
            W4s[i] = (k < CNN_K) ? w1[(ci * 2 + co) * CNN_K + k] : 0.0f;
        }
    }
    if (tid < CNN_C) Bs[tid] = bias[tid];
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the weights were written with generic stores
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    // layer 2 tiles: t0 = T.row0(j); layer 3 tiles: t0 = T.row0(j) - 1
    const int n_jobs = T.n_jobs;

    // ---- LAYER 2 tile building by the workers: x window -> layer 1 on the FP32 pipe -> hi / lo planes of buffer b ----
    float px[2];
    float w1r[8][CNN_K], b1r[8];  // layer-1 weights of this warp's channel octet
    if (LAYER == 2 && warp < TC_WORKERS / 32) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            b1r[j] = W1s[CNN_C * CNN_K + warp * 8 + j];
#pragma unroll
            for (int k = 0; k < CNN_K; k++) w1r[j][k] = W1s[(warp * 8 + j) * CNN_K + k];
        }
    }
    auto prefetch = [&](int job) {
        // x of row t0 - 3 (packed: 3 (t0 - 3) - 3 = 3 t0 - 12 in the whole chunk's x; per-read: in its read's x row).
        // Samples of other reads that land in the window only feed rows that are not positions of this tile's reads.
        const int x0 = (job / T.jpr) * Lx + 3 * ((job % T.jpr) * TC_ROWS) - 12, xn = n_reads * Lx;
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int i = tid + u * TC_WORKERS, j = x0 + i;
            px[u] = (i < TC_NX && j >= 0 && j < xn) ? ((const float *)in)[j] : 0.0f;
        }
    };
    auto build = [&](int job, int b) {
        const int t0 = T.row0(job);
        unsigned char *hi_plane = Abuf + (size_t)b * 2 * TC_PLANE, *lo_plane = hi_plane + TC_PLANE;
        asm volatile("bar.sync 1, %0;" ::"n"(TC_WORKERS) : "memory");  // every worker is done with the previous x window
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int i = tid + u * TC_WORKERS;
            if (i < TC_NX) Xs[i] = px[u];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_WORKERS) : "memory");
        // warp w builds channel octet w (its 8 x 7 layer-1 weights live in registers), lanes walk the rows
        for (int q = lane; q < TC_NQ; q += 32) {
            int r, p;
            float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // zero padding of layer 2's input outside the reads
            if (tc_row_read(t0 - 3 + q, T.S, L1, n_reads, r, p)) {
                float xs[CNN_K];
#pragma unroll
                for (int k = 0; k < CNN_K; k++) xs[k] = Xs[3 * q + k];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    float a = b1r[j];
#pragma unroll
                    for (int k = 0; k < CNN_K; k++) a = fmaf(w1r[j][k], xs[k], a);
                    v[j] = fmaxf(a, 0.0f);
                }
            }
            // (only a position of a read can leave the range: r is that read)
            if (tc_split_store(hi_plane, lo_plane, warp, q, v)) { redo[r] = 1; redo[-1] = 1; }  // redo[-1]: "any read flagged" (lets the FP32 pass leave at once)
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> visible to the tensor core
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&afull[b])) : "memory");
    };
    // ---- LAYER 3 tile loading: sixteen bulk copies (plane x octet runs of 134 rows) completing on afull[b] ----
    auto load_tile = [&](int job, int b) {
        // rows t0 - 3 .. t0 + 130 with t0 = row0 - 1: rho = g + 4 starts at row0
        const unsigned char *src = (const unsigned char *)in + (size_t)T.row0(job) * 16;
        unsigned char *dst = Abuf + (size_t)b * 2 * TC_PLANE;
        mbar_expect_tx(&afull[b], 16 * TC_TILE_RUN);
#pragma unroll 1
        for (int pk = 0; pk < 16; pk++)  // pk = plane * 8 + octet
            tma_bulk_g2s(dst + (size_t)pk * (TC_RA * 16), src + (size_t)pk * ((size_t)a0t_rows * 16), TC_TILE_RUN, &afull[b]);
    };
    // ---- the 56 MMAs of one tile: 7 taps x 4 K-steps of 16 channels x { A_hi x [W_hi | W_lo] (N = 128), A_lo x W_hi
    // (N = 64) }.  Columns 0 .. 63 of the accumulator collect hi * hi + lo * hi, columns 64 .. 127 hi * lo (added by the
    // epilogue).  Three separate N = 64 products read 18 KB of operands from shared memory per tap and K-step -- more
    // than the SM's shared memory delivers in the 96 cycles the tensor core needs for them (the kernels were bound by
    // exactly that: tensor pipe 55 - 61 % active); side by side the activation tile is read once for two products: 14 KB.
    const uint32_t w_lo0 = tc_desc_lo(smem_u32(Wsm), 128 * 16), w_hi = tc_desc_hi(128);
    const uint32_t a_hi_word = tc_desc_hi(128);
    auto issue = [&](int sb, int tb) {
        const uint32_t ah0 = tc_desc_lo(smem_u32(Abuf + (size_t)sb * 2 * TC_PLANE), TC_RA * 16);
        const uint32_t al0 = ah0 + (TC_PLANE >> 4);
        const uint32_t d = tmem + (uint32_t)(tb * 128);
#pragma unroll
        for (int k = 0; k < CNN_K; k++) {
#pragma unroll
            for (int kp = 0; kp < 4; kp++) {
                const uint32_t a_off = (uint32_t)((2 * kp) * TC_RA + k);              // 16-byte units
                const uint32_t w_off = (uint32_t)(((k * 2) * TC_WPART + 2 * kp * 128 * 16) >> 4);  // (tap, octet 2 kp): hi rows, lo rows
                tc_mma_f16(d, ah0 + a_off, a_hi_word, w_lo0 + w_off, w_hi, (k > 0 || kp > 0) ? 1u : 0u, TC_IDESC2);
                tc_mma_f16(d, al0 + a_off, a_hi_word, w_lo0 + w_off, w_hi, 1u, TC_IDESC);
            }
        }
        tc_commit(&accb[tb]);
    };
    // ---- epilogue of one tile: warp w reads TMEM lanes (w % 4) * 32.., columns (w / 4) * 32.. of accumulator tb ----
    auto epilogue = [&](int job, int tb, uint32_t phase, int eb) {
        const int g = T.row0(job) - (LAYER == 3 ? 1 : 0) + (warp & 3) * 32 + lane;  // this thread's row
        mbar_wait(&accb[tb], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = (warp & 3) * 32 + lane, ch0 = ((warp >> 2) & 1) * 32;  // (layer 2: the drainers are warps 8 .. 15)
        int r, p;
        // rows that are not positions of a read are zero padding: for layer 3's input and for the transposed convolution
        const bool live = tc_row_read(g, T.S, L1, n_reads, r, p);
        uint32_t v[32];
        if (LAYER == 3) {
            const int co = warp >> 2, wq = warp & 3;
            const uint32_t taddr = tmem + ((uint32_t)(wq * 32) << 16) + (uint32_t)(tb * 128);
            float P[CNN_K] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            const float4 *wv = reinterpret_cast<const float4 *>(W4s + co * 512);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                tc_ld32(taddr + (uint32_t)(hh * 32), v);
                {   // + the hi * lo products (columns 64 ..)
                    uint32_t v2[32];
                    tc_ld32(taddr + (uint32_t)(64 + hh * 32), v2);
#pragma unroll
                    for (int c = 0; c < 32; c++) v[c] = __float_as_uint(__fadd_rn(__uint_as_float(v[c]), __uint_as_float(v2[c])));
                }
                if (hh == 1) {  // both halves are in registers: hand the accumulator back
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&accfree[tb])) : "memory");
                }
                if (CSLOT >= 0) {
                    // weights and biases from the constant bank; with the slot a template parameter and the branch on co
                    // (uniform per warp) every address is a compile-time constant: the FFMAs / FADDs take their second
                    // operand straight from the bank (c[3][imm]), no load instruction at all
                    auto acc = [&](const float *cw, const float *cb) {
#pragma unroll
                        for (int c = 0; c < 32; c++) {
                            const int ci = hh * 32 + c;
                            const float a = live ? fmaxf(__fadd_rn(__uint_as_float(v[c]), cb[ci]), 0.0f) : 0.0f;
#pragma unroll
                            for (int j = 0; j < CNN_K; j++) P[j] = fmaf(a, cw[ci * 8 + j], P[j]);
                        }
                    };
                    constexpr int SL = CSLOT >= 0 ? CSLOT : 0;
                    if (co == 0) acc(&adb_c_convT[SL][0], &adb_c_convT[SL][1024]);
                    else acc(&adb_c_convT[SL][512], &adb_c_convT[SL][1024]);
                } else {
#pragma unroll
                    for (int c = 0; c < 32; c++) {
                        const int ci = hh * 32 + c;
                        const float a = live ? fmaxf(__fadd_rn(__uint_as_float(v[c]), Bs[ci]), 0.0f) : 0.0f;
                        const float4 w0 = wv[ci * 2], w1v = wv[ci * 2 + 1];
                        P[0] = fmaf(a, w0.x, P[0]); P[1] = fmaf(a, w0.y, P[1]); P[2] = fmaf(a, w0.z, P[2]); P[3] = fmaf(a, w0.w, P[3]);
                        P[4] = fmaf(a, w1v.x, P[4]); P[5] = fmaf(a, w1v.y, P[5]); P[6] = fmaf(a, w1v.z, P[6]);
                    }
                }
            }
            // neighbours: P0..P2 of row q + 1, P6 of row q - 1
            float up0 = __shfl_down_sync(ADB_FULL, P[0], 1), up1 = __shfl_down_sync(ADB_FULL, P[1], 1);
            float up2 = __shfl_down_sync(ADB_FULL, P[2], 1), dn6 = __shfl_up_sync(ADB_FULL, P[6], 1);
            float *eg = Eg + ((eb * 2 + co) * 4) * 4;
            if (lane == 0) { eg[wq * 4 + 0] = P[0]; eg[wq * 4 + 1] = P[1]; eg[wq * 4 + 2] = P[2]; }
            if (lane == 31) eg[wq * 4 + 3] = P[6];
            asm volatile("bar.sync 1, %0;" ::"n"(TC_WORKERS) : "memory");
            if (lane == 31 && wq < 3) { up0 = eg[(wq + 1) * 4 + 0]; up1 = eg[(wq + 1) * 4 + 1]; up2 = eg[(wq + 1) * 4 + 2]; }
            if (lane == 0 && wq > 0) dn6 = eg[(wq - 1) * 4 + 3];
            const int Lout = Lx;
            if (q >= 1 && q <= TC_L3_STRIDE && live && 3 * p < Lout) {
                const float bco = b1[co];
                float *orow = (float *)out + ((size_t)r * 2 + co) * Lout + 3 * p;
                orow[0] = __fadd_rn(bco, __fadd_rn(__fadd_rn(up0, P[3]), dn6));
                if (3 * p + 1 < Lout) orow[1] = __fadd_rn(bco, __fadd_rn(up1, P[4]));
                if (3 * p + 2 < Lout) orow[2] = __fadd_rn(bco, __fadd_rn(up2, P[5]));
            }
        } else {
            // bias + ReLU, split, and straight into layer 3's tile layout (rows outside the reads: zeros = its padding)
            const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(tb * 128 + ch0);
            tc_ld32(taddr, v);
            {   // + the hi * lo products (columns 64 ..)
                uint32_t v2[32];
                tc_ld32(taddr + 64u, v2);
#pragma unroll
                for (int c = 0; c < 32; c++) v[c] = __float_as_uint(__fadd_rn(__uint_as_float(v[c]), __uint_as_float(v2[c])));
            }
            unsigned char *base = (unsigned char *)out + (size_t)(g + TC_A0T_PAD) * 16;
            bool bad = false;
#pragma unroll
            for (int o = 0; o < 4; o++) {
                __half2 h[4], l[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    float f0 = fmaxf(__fadd_rn(__uint_as_float(v[8 * o + 2 * j]), Bs[ch0 + 8 * o + 2 * j]), 0.0f);
                    float f1 = fmaxf(__fadd_rn(__uint_as_float(v[8 * o + 2 * j + 1]), Bs[ch0 + 8 * o + 2 * j + 1]), 0.0f);
                    if (!live) { f0 = 0.0f; f1 = 0.0f; }
                    const __half h0 = __float2half_rn(f0), h1 = __float2half_rn(f1);
                    const float g0 = __half2float(h0), g1 = __half2float(h1);
                    bad |= !(fabsf(g0) <= 65504.0f) || !(fabsf(g1) <= 65504.0f);
                    h[j] = __halves2half2(h0, h1);
                    l[j] = __halves2half2(__float2half_rn(__fsub_rn(f0, g0)), __float2half_rn(__fsub_rn(f1, g1)));
                }
                const size_t off = (size_t)((ch0 >> 3) + o) * ((size_t)a0t_rows * 16);
                *reinterpret_cast<uint4 *>(base + off) = *reinterpret_cast<const uint4 *>(h);
                *reinterpret_cast<uint4 *>(base + (size_t)8 * ((size_t)a0t_rows * 16) + off) = *reinterpret_cast<const uint4 *>(l);
            }
            if (bad) { redo[r] = 1; redo[-1] = 1; }  // (gap rows are zeros: a flagged row is a position of read r)
        }
    };

    if (warp == NWW) {
        // ---- MMA issuer ----
        if (tc_elect_one()) {
            uint32_t it = 0;
            for (int job = blockIdx.x; job < n_jobs; job += gridDim.x, it++) {
                const int tb = (int)(it & 1u), sb = (int)(it % NBUF);
                mbar_wait(&afull[sb], (it / NBUF) & 1u);                       // tile buffer ready
                if (it >= 2) mbar_wait(&accfree[tb], ((it - 2) >> 1) & 1u);    // accumulator drained (tile it - 2)
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue(sb, tb);
                if (LAYER == 3) tc_commit(&sfree[sb]);                         // tile buffer free once these MMAs are done
            }
        }
        __syncwarp();
    } else if (warp == NWW + 1) {
        // ---- tile loader (layer 3): runs up to NBUF tiles ahead; tile it reuses the buffer of tile it - NBUF, whose
        // next release needs the tile loaded here, so the parity wait cannot be overtaken ----
        if (LAYER == 3 && lane == 0) {
            uint32_t it = 0;
            for (int job = blockIdx.x; job < n_jobs; job += gridDim.x, it++) {
                const int sb = (int)(it % NBUF);
                if (it >= NBUF) mbar_wait(&sfree[sb], ((it / NBUF) - 1) & 1u);
                load_tile(job, sb);
            }
        }
        __syncwarp();
    } else {
        // ---- workers ----
        if (LAYER == 2) {
            // Layer 2 splits its workers: warps 0 .. 7 BUILD the operand tiles (x window -> layer 1 -> hi / lo planes),
            // warps 8 .. 15 DRAIN the accumulators (bias + ReLU + split -> A0T).  Both loops run side by side, so a tile
            // costs max(build, drain) instead of their sum (the tensor pipe was idle 45 % of the time behind eight
            // warps doing both).  A tile buffer is rebuilt once the MMAs that read it are complete: the builders wait on
            // the same accumulator barrier as the drainers (parity waits do not consume it).
            if (warp < TC_WORKERS / 32) {
                // (the x window of a tile is loaded into registers a whole tile ahead of the build that consumes it)
                int job = blockIdx.x;
                if (job < n_jobs) {
                    prefetch(job);
                    build(job, 0);
                    if (job + (int)gridDim.x < n_jobs) prefetch(job + (int)gridDim.x);
                }
                uint32_t it = 0;
                for (; job < n_jobs; job += gridDim.x, it++) {
                    const int b = (int)(it & 1u);
                    const int next = job + (int)gridDim.x;
                    if (next < n_jobs) {
                        if (it >= 1) mbar_wait(&accb[b ^ 1], ((it - 1) >> 1) & 1u);  // tile it - 1 (buffer b ^ 1) has been multiplied
                        build(next, b ^ 1);
                        if (next + (int)gridDim.x < n_jobs) prefetch(next + (int)gridDim.x);
                    }
                }
            } else {
                uint32_t it = 0;
                for (int job = blockIdx.x; job < n_jobs; job += gridDim.x, it++) {
                    const int tb = (int)(it & 1u);
                    epilogue(job, tb, (it >> 1) & 1u, tb);
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&accfree[tb])) : "memory");
                }
            }
        } else {
            int prev_job = -1;
            uint32_t it = 0;
            for (int job = blockIdx.x; job < n_jobs; job += gridDim.x, it++) {
                const int b = (int)(it & 1u);
                if (prev_job >= 0) epilogue(prev_job, b ^ 1, ((it - 1) >> 1) & 1u, b ^ 1);  // (hands the accumulator back itself)
                prev_job = job;
            }
            if (prev_job >= 0) epilogue(prev_job, (int)((it - 1) & 1u), ((it - 1) >> 1) & 1u, (int)((it - 1) & 1u));
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256));
}

static int cnn_tc_launch_setup() {
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(2)) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(3)) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<3, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(3)) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(3)) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(3)) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(cnn_conv64_tc_kernel<3, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cnn_tc_smem_bytes_layer(3)) != cudaSuccess) return -1;
    return 0;
}

// layer 2: in = x, out = A0T;  layer 3: in = A0T, out = scores [N][2][Lout] (w1 / b1 = W4 / b4, Lx = Lout)
static void cnn_tc_launch(int layer, const void *in, void *out, const __half *wp, const float *bias, const float *w1,
                          const float *b1, int n_reads, int Lx, int L1, int LP, int per_read, int *redo, int sm_count,
                          cudaStream_t st, int cslot) {
    const int jobs = cnn_tc_tiles(layer, n_reads, L1, per_read).n_jobs;
    const int grid = std::max(1, std::min(jobs, sm_count));
    const size_t smem = cnn_tc_smem_bytes_layer(layer);
    if (layer == 2) cnn_conv64_tc_kernel<2><<<grid, TC_THREADS2, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
    else if (cslot == 0) cnn_conv64_tc_kernel<3, 0><<<grid, TC_THREADS, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
    else if (cslot == 1) cnn_conv64_tc_kernel<3, 1><<<grid, TC_THREADS, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
    else if (cslot == 2) cnn_conv64_tc_kernel<3, 2><<<grid, TC_THREADS, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
    else if (cslot == 3) cnn_conv64_tc_kernel<3, 3><<<grid, TC_THREADS, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
    else cnn_conv64_tc_kernel<3><<<grid, TC_THREADS, smem, st>>>(in, out, wp, bias, w1, b1, n_reads, Lx, L1, LP, per_read, redo);
}

static int cnn_tc_a0t_rows_host(int n_reads, int L1, int per_read) { return cnn_tc_a0t_rows(n_reads, L1, per_read); }
static int cnn_tc_read_rows_host(int L1, int per_read) { return cnn_tc_read_rows(L1, per_read); }
