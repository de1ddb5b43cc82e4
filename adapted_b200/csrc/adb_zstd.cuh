// Device-side zstd decode (RFC 8878, frames without dictionaries): the zstd stage of pod5's VBZ, so that compressed
// reads cross PCIe as frames and svb16_decode_kernel (adb_svb16.cuh) takes the decoded streams from HBM.
//
// One WARP per frame, grid-striding.  Lane 0 parses the frame and block headers, builds the tables and decodes the
// sequences in batches of ZSTDG_SEQ_BATCH into shared memory; the warp then executes a batch (literal copies and match
// copies, one sequence after the other, all lanes on the bytes of one copy).  A match byte j of a copy with offset o
// is out[j % o - o]: every byte of a copy reads bytes produced before the copy started, so all lanes copy at once
// whatever the offset (offsets 1-3 included) and only consecutive sequences are ordered (__syncwarp).  Huffman
// literals of a 4-stream block are decoded by lanes 0-3, one stream each; the XXH64 checksum runs its four
// accumulators on lanes 0-3.
//
// Decoded literals are parked at the END of the frame's output slot (as libzstd does when the block fits): the write
// position never passes the next unread literal while the block's output fits the slot, and a block whose output does
// not fit fails with ZSTDG_E_DST_SIZE.  So the decoder needs no scratch memory beyond shared memory.
//
// Memory safety: every bit-reader load is clamped to the frame's bytes (a byte outside reads as zero; the callers need
// no slack behind a frame), every write is checked against the slot [dst_off[i], dst_off[i] + dst_cap[i]), and every
// match source against the bytes produced.  A malformed frame ends with a negative status, never an access outside
// its frame or its slot.
#pragma once
#include "adb_common.cuh"

// status codes (negative; a decoded frame's status is its decoded size)
#define ZSTDG_E_TRUNCATED (-1)   // the frame ends before its last block, or a section runs past its block
#define ZSTDG_E_MAGIC (-2)       // not a zstd frame (skippable frames included)
#define ZSTDG_E_RESERVED (-3)    // a reserved bit or a reserved block / literals / sequence mode is set
#define ZSTDG_E_DICT (-4)        // dictionary ID other than 0
#define ZSTDG_E_DST_SIZE (-5)    // output past the slot's capacity, or a block past the block maximum
#define ZSTDG_E_OFFSET (-6)      // match offset beyond the bytes produced or beyond the window
#define ZSTDG_E_SIZE (-7)        // decoded size differs from the frame's content size
#define ZSTDG_E_CHECKSUM (-8)    // XXH64 content checksum mismatch
#define ZSTDG_E_CORRUPT (-9)     // a table description or a bitstream RFC 8878 declares corrupt
#define ZSTDG_E_TRAILING (-10)   // bytes left over behind the last block (and checksum)

#define ZSTDG_THREADS 128
#define ZSTDG_SEQ_BATCH 128
#define ZSTDG_HUF_LOG 11

struct ZstdArgs {
    const uint8_t *src;       // frames
    const int64_t *src_off;   // [n + 1] frame i = src[src_off[i] .. src_off[i + 1])
    uint8_t *dst;
    const int64_t *dst_off;   // [n] slot start of every frame
    const int64_t *dst_cap;   // [n] slot size, or nullptr: dst_off[i + 1] - dst_off[i]
    int32_t *status;          // [n]
    int32_t *n_failed;        // optional: frames with a negative status are counted here
    int n;
};

// per-warp shared memory
struct ZstdSmem {
    uint16_t huf[1 << ZSTDG_HUF_LOG];   // symbol | nbBits << 8
    uint32_t ll[512], of[256], ml[512];  // FSE cells: symbol | nbBits << 8 | baseline << 16
    uint32_t wt[64];                     // FSE table of the Huffman weights
    uint32_t seq_ll[ZSTDG_SEQ_BATCH], seq_ml[ZSTDG_SEQ_BATCH], seq_of[ZSTDG_SEQ_BATCH];
    uint8_t weights[256];
    uint16_t hstart[256];
    int16_t norm[64];
    int32_t sh[16];                      // broadcast of lane 0's decisions
};

namespace zstdg {

__device__ __forceinline__ int highbit(uint32_t v) { return 31 - __clz(v); }

// backward bitstream (Huffman streams, FSE streams): bits are consumed from the end; `pos` = bits left, may go
// negative (bits below the start read as zero), which a decoder reports as corruption where it matters
struct BitB {
    const uint8_t *s;
    int len;
    int pos;
    uint64_t c;
    int cb;  // the container holds stream bits [cb, cb + 64)
    __device__ __forceinline__ void refill() {
        cb = ((pos - 57) >> 3) << 3;  // floor to a byte; pos - cb in [57, 64]
        const int b0 = cb >> 3;
        uint64_t v = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int b = b0 + k;
            const uint64_t x = (b >= 0 && b < len) ? (uint64_t)__ldg(s + b) : 0ull;
            v |= x << (8 * k);
        }
        c = v;
    }
    // 0: ok, 1: empty stream or no end marker
    __device__ __forceinline__ int init(const uint8_t *p, int n) {
        s = p; len = n;
        if (n <= 0) return 1;
        const uint8_t last = p[n - 1];
        if (last == 0) return 1;
        pos = (n - 1) * 8 + highbit(last);
        refill();
        return 0;
    }
    __device__ __forceinline__ uint32_t peek(int nb) {  // nb <= 32
        if (pos - nb < cb) refill();
        return nb ? (uint32_t)((c >> (pos - nb - cb)) & ((1ull << nb) - 1ull)) : 0u;
    }
    __device__ __forceinline__ void skip(int nb) { pos -= nb; }
    __device__ __forceinline__ uint32_t read(int nb) { const uint32_t v = peek(nb); pos -= nb; return v; }
};

// forward little-endian reader of an FSE table description; bytes beyond `len` read as zero
struct BitF {
    const uint8_t *s;
    int len;
    int pos;  // bits consumed
    __device__ __forceinline__ uint32_t peek(int nb) {  // nb <= 24
        const int b0 = pos >> 3;
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { const int b = b0 + k; v |= (b < len ? (uint32_t)s[b] : 0u) << (8 * k); }
        return (v >> (pos & 7)) & ((1u << nb) - 1u);
    }
};

// RFC 8878 4.1.1: normalized counts from a table description; returns the bytes used, or -1
__device__ int read_ncount(const uint8_t *p, int avail, int max_log, int max_sym, int16_t *norm, int *log_out, int *nsym_out) {
    BitF b{p, avail, 0};
    const int al = (int)b.peek(4) + 5;
    b.pos += 4;
    if (al > max_log) return -1;
    int remaining = (1 << al) + 1, threshold = 1 << al, nb = al + 1, sym = 0;
    bool prev0 = false;
    for (;;) {
        if (prev0) {
            int r;
            do {
                r = (int)b.peek(2);
                b.pos += 2;
                for (int k = 0; k < r; k++) { if (sym > max_sym) return -1; norm[sym++] = 0; }
            } while (r == 3);
        }
        if (sym > max_sym) return -1;
        const int mx = (2 * threshold - 1) - remaining;
        int count;
        const uint32_t low = b.peek(nb - 1);
        if ((int)(low & (threshold - 1)) < mx) {
            count = (int)(low & (threshold - 1));
            b.pos += nb - 1;
        } else {
            count = (int)b.peek(nb) & (2 * threshold - 1);
            if (count >= threshold) count -= mx;
            b.pos += nb;
        }
        count--;
        remaining -= count < 0 ? -count : count;
        norm[sym++] = (int16_t)count;
        prev0 = count == 0;
        if (remaining <= 1) break;
        while (remaining < threshold) { nb--; threshold >>= 1; }
        if (sym > max_sym) return -1;
        if (b.pos > avail * 8) return -1;
    }
    if (remaining != 1) return -1;
    const int used = (b.pos + 7) >> 3;
    if (used > avail) return -1;
    *log_out = al;
    *nsym_out = sym;
    return used;
}

// RFC 8878 4.1.1: decoding table from normalized counts (one lane); 0 ok, -1 corrupt
__device__ int build_fse(uint32_t *tab, const int16_t *norm, int nsym, int al) {
    const int size = 1 << al, mask = size - 1;
    int high = size - 1;
    uint16_t next[64];
    for (int s = 0; s < nsym; s++) {
        if (norm[s] == -1) { tab[high--] = (uint32_t)s; next[s] = 1; }
        else next[s] = (uint16_t)norm[s];
    }
    const int step = (size >> 1) + (size >> 3) + 3;
    int pos = 0;
    for (int s = 0; s < nsym; s++)
        for (int i = 0; i < norm[s]; i++) {
            tab[pos] = (uint32_t)s;
            do { pos = (pos + step) & mask; } while (pos > high);
        }
    if (pos != 0) return -1;
    for (int u = 0; u < size; u++) {
        const int s = (int)(tab[u] & 0xffu);
        const int ns = next[s]++;
        const int nbits = al - highbit((uint32_t)ns);
        const int base = (ns << nbits) - size;
        tab[u] = (uint32_t)s | ((uint32_t)nbits << 8) | ((uint32_t)base << 16);
    }
    return 0;
}

__constant__ int16_t c_ll_def[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
__constant__ int16_t c_ml_def[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                     1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
__constant__ int16_t c_of_def[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
__constant__ uint32_t c_ll_base[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40,
                                       48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
__constant__ uint8_t c_ll_bits[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
__constant__ uint32_t c_ml_base[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29,
                                       30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195,
                                       16387, 32771, 65539};
__constant__ uint8_t c_ml_bits[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                      0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

// one sequence table (LL / OF / ML) by its mode; returns bytes used, or a negative status
__device__ int seq_table(int mode, const uint8_t *p, int avail, uint32_t *tab, int *al, bool *have, int max_log, int max_sym,
                         const int16_t *def, int def_n, int def_log, int16_t *norm) {
    if (mode == 0) {
        for (int s = 0; s < def_n; s++) norm[s] = def[s];
        if (build_fse(tab, norm, def_n, def_log)) return ZSTDG_E_CORRUPT;
        *al = def_log;
        *have = true;
        return 0;
    }
    if (mode == 1) {
        if (avail < 1) return ZSTDG_E_TRUNCATED;
        if (p[0] > max_sym) return ZSTDG_E_CORRUPT;
        tab[0] = (uint32_t)p[0];  // nbBits 0, baseline 0
        *al = 0;
        *have = true;
        return 1;
    }
    if (mode == 2) {
        int lg, ns;
        const int used = read_ncount(p, avail, max_log, max_sym, norm, &lg, &ns);
        if (used < 0) return ZSTDG_E_CORRUPT;
        if (build_fse(tab, norm, ns, lg)) return ZSTDG_E_CORRUPT;
        *al = lg;
        *have = true;
        return used;
    }
    return *have ? 0 : ZSTDG_E_CORRUPT;  // repeat: the previous block's table of this frame
}

__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
#define XP1 11400714785074694791ull
#define XP2 14029467366897019727ull
#define XP3 1609587929392839161ull
#define XP4 9650029242287828579ull
#define XP5 2870177450012600261ull
__device__ __forceinline__ uint64_t xround(uint64_t acc, uint64_t in) { acc += in * XP2; acc = rotl64(acc, 31); return acc * XP1; }
__device__ __forceinline__ uint64_t xmerge(uint64_t acc, uint64_t v) { acc ^= xround(0, v); return acc * XP1 + XP4; }
__device__ __forceinline__ uint64_t ld64(const uint8_t *p) {
    uint64_t v = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) v |= (uint64_t)p[k] << (8 * k);
    return v;
}

// XXH64 (seed 0) of p[0 .. len) by the warp: lanes 0-3 run the four stripe accumulators; the result is valid on all lanes
__device__ uint64_t xxh64_warp(const uint8_t *p, int64_t len, int lane) {
    const int64_t nstripes = len >> 5;
    uint64_t v = lane == 0 ? XP1 + XP2 : lane == 1 ? XP2 : lane == 2 ? 0ull : 0ull - XP1;
    if (lane < 4)
        for (int64_t i = 0; i < nstripes; i++) v = xround(v, ld64(p + 32 * i + 8 * lane));
    const uint64_t v1 = __shfl_sync(ADB_FULL, v, 0), v2 = __shfl_sync(ADB_FULL, v, 1), v3 = __shfl_sync(ADB_FULL, v, 2),
                   v4 = __shfl_sync(ADB_FULL, v, 3);
    uint64_t h;
    if (len >= 32) {
        h = rotl64(v1, 1) + rotl64(v2, 7) + rotl64(v3, 12) + rotl64(v4, 18);
        h = xmerge(h, v1); h = xmerge(h, v2); h = xmerge(h, v3); h = xmerge(h, v4);
    } else {
        h = XP5;
    }
    h += (uint64_t)len;
    int64_t i = nstripes << 5;
    for (; i + 8 <= len; i += 8) { h ^= xround(0, ld64(p + i)); h = rotl64(h, 27) * XP1 + XP4; }
    if (i + 4 <= len) {
        const uint64_t w = (uint64_t)p[i] | ((uint64_t)p[i + 1] << 8) | ((uint64_t)p[i + 2] << 16) | ((uint64_t)p[i + 3] << 24);
        h ^= w * XP1; h = rotl64(h, 23) * XP2 + XP3; i += 4;
    }
    for (; i < len; i++) { h ^= (uint64_t)p[i] * XP5; h = rotl64(h, 11) * XP1; }
    h ^= h >> 33; h *= XP2; h ^= h >> 29; h *= XP3; h ^= h >> 32;
    return h;
}

// Huffman tree description (RFC 8878 4.2.1) -> decoding table in S.huf; returns bytes used, or a negative status.
// Lane 0 reads the weights; the warp fills the table.  *max_bits receives the table log.
__device__ int read_huffman(ZstdSmem &S, const uint8_t *p, int avail, int lane, int *max_bits) {
    int nw = 0, used = 0, rc = 0;
    if (lane == 0) {
        do {
            if (avail < 1) { rc = ZSTDG_E_TRUNCATED; break; }
            const int hb = p[0];
            if (hb >= 128) {
                nw = hb - 127;
                used = 1 + (nw + 1) / 2;
                if (used > avail) { rc = ZSTDG_E_TRUNCATED; break; }
                for (int k = 0; k < nw; k++) S.weights[k] = (uint8_t)((p[1 + k / 2] >> ((k & 1) ? 0 : 4)) & 15);
            } else {
                used = 1 + hb;
                if (used > avail || hb == 0) { rc = ZSTDG_E_TRUNCATED; break; }
                int lg, ns;
                const int hu = read_ncount(p + 1, hb, 6, 12, S.norm, &lg, &ns);
                if (hu < 0 || build_fse(S.wt, S.norm, ns, lg)) { rc = ZSTDG_E_CORRUPT; break; }
                BitB b;
                if (b.init(p + 1 + hu, hb - hu)) { rc = ZSTDG_E_CORRUPT; break; }
                uint32_t s1 = b.read(lg), s2 = b.read(lg);
                for (;;) {
                    if (nw > 253) { rc = ZSTDG_E_CORRUPT; break; }
                    uint32_t e = S.wt[s1];
                    S.weights[nw++] = (uint8_t)(e & 0xff);
                    s1 = (e >> 16) + b.read((e >> 8) & 0xff);
                    if (b.pos < 0) { S.weights[nw++] = (uint8_t)(S.wt[s2] & 0xff); break; }
                    e = S.wt[s2];
                    S.weights[nw++] = (uint8_t)(e & 0xff);
                    s2 = (e >> 16) + b.read((e >> 8) & 0xff);
                    if (b.pos < 0) { S.weights[nw++] = (uint8_t)(S.wt[s1] & 0xff); break; }
                }
                if (rc) break;
            }
            // the last symbol's weight is implied: the weights fill a power of two
            uint32_t total = 0;
            for (int k = 0; k < nw; k++) {
                if (S.weights[k] > ZSTDG_HUF_LOG) { rc = ZSTDG_E_CORRUPT; break; }
                if (S.weights[k]) total += 1u << (S.weights[k] - 1);
            }
            if (rc) break;
            if (total == 0) { rc = ZSTDG_E_CORRUPT; break; }
            const int mb = highbit(total) + 1;
            const uint32_t rest = (1u << mb) - total;
            if (mb > ZSTDG_HUF_LOG || (rest & (rest - 1)) != 0 || nw > 255) { rc = ZSTDG_E_CORRUPT; break; }
            S.weights[nw++] = (uint8_t)(highbit(rest) + 1);
            // table ranges: symbols of weight w take 2^(w-1) cells each, weights in increasing order
            uint32_t rank[ZSTDG_HUF_LOG + 2];
            for (int w = 0; w <= ZSTDG_HUF_LOG + 1; w++) rank[w] = 0;
            for (int k = 0; k < nw; k++) rank[S.weights[k]]++;
            uint32_t start = 0;
            for (int w = 1; w <= mb; w++) { const uint32_t c = rank[w] << (w - 1); rank[w] = start; start += c; }
            for (int k = 0; k < nw; k++) {
                const int w = S.weights[k];
                S.hstart[k] = (uint16_t)(w ? rank[w] : 0);
                if (w) rank[w] += 1u << (w - 1);
            }
            S.sh[1] = mb;
        } while (0);
        S.sh[0] = rc ? rc : used;
        S.sh[2] = nw;
    }
    __syncwarp();
    rc = S.sh[0];
    if (rc < 0) return rc;
    const int mb = S.sh[1];
    nw = S.sh[2];
    for (int k = lane; k < nw; k += 32) {
        const int w = S.weights[k];
        if (!w) continue;
        const int n = 1 << (w - 1), st = S.hstart[k];
        const uint16_t e = (uint16_t)(k | ((mb + 1 - w) << 8));
        for (int j = 0; j < n; j++) S.huf[st + j] = e;
    }
    __syncwarp();
    *max_bits = mb;
    return rc;
}

// one Huffman stream of `cnt` symbols into out; 0 ok, else corrupt
__device__ int huf_stream(const ZstdSmem &S, int mb, const uint8_t *p, int len, uint8_t *out, int cnt) {
    BitB b;
    if (b.init(p, len)) return 1;
    for (int k = 0; k < cnt; k++) {
        const uint16_t e = S.huf[b.peek(mb)];
        out[k] = (uint8_t)(e & 0xff);
        b.skip(e >> 8);
    }
    return b.pos != 0;
}

}  // namespace zstdg

// the kernel's dynamic shared memory
#define ZSTDG_SMEM ((ZSTDG_THREADS / 32) * sizeof(ZstdSmem))

__global__ void __launch_bounds__(ZSTDG_THREADS) zstd_decode_kernel(ZstdArgs A) {
    using namespace zstdg;
    extern __shared__ __align__(16) uint8_t zsm[];
    const int lane = threadIdx.x & 31;
    ZstdSmem &S = reinterpret_cast<ZstdSmem *>(zsm)[threadIdx.x >> 5];
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int fi = warp; fi < A.n; fi += nwarps) {
        const uint8_t *src = A.src + A.src_off[fi];
        const int64_t slen = A.src_off[fi + 1] - A.src_off[fi];
        uint8_t *dst = A.dst + A.dst_off[fi];
        const int64_t cap = A.dst_cap ? A.dst_cap[fi] : A.dst_off[fi + 1] - A.dst_off[fi];
        int64_t produced = 0;
        int status = 0;
        // ---- frame header (every lane parses it: a handful of bytes) ----
        int64_t ip = 0, content = -1;
        uint64_t window = 0;
        bool checksum = false;
        do {
            if (slen < 6) { status = ZSTDG_E_TRUNCATED; break; }
            const uint32_t magic = (uint32_t)src[0] | ((uint32_t)src[1] << 8) | ((uint32_t)src[2] << 16) | ((uint32_t)src[3] << 24);
            if (magic != 0xFD2FB528u) { status = ZSTDG_E_MAGIC; break; }
            const int fhd = src[4];
            const int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
            if (fhd & 8) { status = ZSTDG_E_RESERVED; break; }
            checksum = (fhd >> 2) & 1;
            ip = 5;
            if (!single) {
                const int wd = src[ip++];
                const int e = wd >> 3, mnt = wd & 7;
                const uint64_t base = 1ull << (10 + e);
                window = base + (base >> 3) * (uint64_t)mnt;
            }
            const int did_sz = did_flag == 3 ? 4 : did_flag;
            const int fcs_sz = fcs_flag == 0 ? single : (1 << fcs_flag);
            if (ip + did_sz + fcs_sz > slen) { status = ZSTDG_E_TRUNCATED; break; }
            uint32_t did = 0;
            for (int k = 0; k < did_sz; k++) did |= (uint32_t)src[ip + k] << (8 * k);
            ip += did_sz;
            if (did != 0) { status = ZSTDG_E_DICT; break; }
            if (fcs_sz) {
                uint64_t v = 0;
                for (int k = 0; k < fcs_sz; k++) v |= (uint64_t)src[ip + k] << (8 * k);
                if (fcs_sz == 2) v += 256;
                ip += fcs_sz;
                content = v > (1ull << 62) ? (int64_t)(1ull << 62) : (int64_t)v;
            }
            if (single) window = (uint64_t)content;
            if (content > cap) status = ZSTDG_E_DST_SIZE;
        } while (0);
        const int64_t block_max = (int64_t)(window < 131072ull ? window : 131072ull);
        const int64_t out_end = cap;  // decoded literals sit at the end of the slot
        int huf_log = 0, ll_log = 0, of_log = 0, ml_log = 0;
        bool have_huf = false, have_ll = false, have_of = false, have_ml = false;
        uint32_t rep[3] = {1, 4, 8};
        bool last = false;
        while (status == 0 && !last) {
            if (ip + 3 > slen) { status = ZSTDG_E_TRUNCATED; break; }
            const uint32_t bh = (uint32_t)src[ip] | ((uint32_t)src[ip + 1] << 8) | ((uint32_t)src[ip + 2] << 16);
            ip += 3;
            last = bh & 1;
            const int btype = (bh >> 1) & 3;
            const int64_t bsize = bh >> 3;
            if (btype == 3) { status = ZSTDG_E_RESERVED; break; }
            if (btype == 1) {  // RLE: one byte, bsize copies
                if (ip + 1 > slen) { status = ZSTDG_E_TRUNCATED; break; }
                if (bsize > block_max || produced + bsize > cap) { status = ZSTDG_E_DST_SIZE; break; }
                const uint8_t v = src[ip];
                for (int64_t j = lane; j < bsize; j += 32) dst[produced + j] = v;
                ip += 1;
                produced += bsize;
                __syncwarp();
                continue;
            }
            if (ip + bsize > slen) { status = ZSTDG_E_TRUNCATED; break; }
            if (btype == 0) {
                if (bsize > block_max || produced + bsize > cap) { status = ZSTDG_E_DST_SIZE; break; }
                for (int64_t j = lane; j < bsize; j += 32) dst[produced + j] = src[ip + j];
                ip += bsize;
                produced += bsize;
                __syncwarp();
                continue;
            }
            // ---- compressed block ----
            // the compressed payload is bounded by 128 KB only (as libzstd checks it); the window bounds the block's
            // decoded size, checked below: a tiny frame's compressed block may be longer than the frame's content
            if (bsize >= 131072) { status = ZSTDG_E_CORRUPT; break; }
            const uint8_t *blk = src + ip;
            const int bl = (int)bsize;
            ip += bsize;
            int q = 0;  // read position in the block
            // literals section header
            if (bl < 1) { status = ZSTDG_E_TRUNCATED; break; }
            const int ltype = blk[0] & 3, lfmt = (blk[0] >> 2) & 3;
            int lit_n = 0, lit_c = 0, nstreams = 1;
            if (ltype < 2) {
                const int hs = (lfmt & 1) == 0 ? 1 : (lfmt == 1 ? 2 : 3);
                if (hs > bl) { status = ZSTDG_E_TRUNCATED; break; }
                if (hs == 1) lit_n = blk[0] >> 3;
                else if (hs == 2) lit_n = (blk[0] >> 4) | (blk[1] << 4);
                else lit_n = (blk[0] >> 4) | (blk[1] << 4) | (blk[2] << 12);
                q = hs;
                lit_c = ltype == 0 ? lit_n : 1;
            } else {
                const int hs = lfmt <= 1 ? 3 : lfmt + 2, nb = lfmt <= 1 ? 10 : (lfmt == 2 ? 14 : 18);
                nstreams = lfmt == 0 ? 1 : 4;
                if (hs > bl) { status = ZSTDG_E_TRUNCATED; break; }
                uint64_t h = 0;
                for (int k = 0; k < hs; k++) h |= (uint64_t)blk[k] << (8 * k);
                lit_n = (int)((h >> 4) & ((1u << nb) - 1u));
                lit_c = (int)((h >> (4 + nb)) & ((1u << nb) - 1u));
                q = hs;
            }
            if (lit_n > block_max) { status = ZSTDG_E_CORRUPT; break; }
            if (q + lit_c > bl) { status = ZSTDG_E_TRUNCATED; break; }
            if (produced + lit_n > cap) { status = ZSTDG_E_DST_SIZE; break; }
            // literals: raw ones are read in place, RLE is one byte, Huffman ones are decoded to the slot's end
            const uint8_t *lit = nullptr;
            uint8_t lit_rle = 0;
            if (ltype == 0) lit = blk + q;
            else if (ltype == 1) lit_rle = blk[q];
            else {
                int hq = q, hused = 0;
                if (ltype == 2) {
                    int mb = 0;
                    hused = read_huffman(S, blk + q, lit_c, lane, &mb);
                    if (hused < 0) { status = hused; break; }
                    huf_log = mb;
                    have_huf = true;
                } else if (!have_huf) { status = ZSTDG_E_CORRUPT; break; }
                hq += hused;
                const int streams_bytes = lit_c - hused;
                uint8_t *lout = dst + (out_end - lit_n);
                int err = 0;
                if (nstreams == 1) {
                    if (lane == 0) err = huf_stream(S, huf_log, blk + hq, streams_bytes, lout, lit_n);
                } else {
                    if (streams_bytes < 10) err = 1;
                    else {
                        const int s1 = blk[hq] | (blk[hq + 1] << 8), s2 = blk[hq + 2] | (blk[hq + 3] << 8), s3 = blk[hq + 4] | (blk[hq + 5] << 8);
                        const int s4 = streams_bytes - 6 - s1 - s2 - s3;
                        const int per = (lit_n + 3) / 4, c4 = lit_n - 3 * per;
                        if (s4 < 1 || c4 < 0) err = 1;
                        else if (lane < 4) {
                            const int soff = hq + 6 + (lane > 0 ? s1 : 0) + (lane > 1 ? s2 : 0) + (lane > 2 ? s3 : 0);
                            const int slen_k = lane == 0 ? s1 : lane == 1 ? s2 : lane == 2 ? s3 : s4;
                            err = huf_stream(S, huf_log, blk + soff, slen_k, lout + lane * per, lane < 3 ? per : c4);
                        }
                    }
                }
                __syncwarp();
                if (__any_sync(ADB_FULL, err)) { status = ZSTDG_E_CORRUPT; break; }
                lit = lout;
            }
            q += lit_c;
            // ---- sequences section ----
            if (q >= bl) { status = ZSTDG_E_TRUNCATED; break; }
            int nseq = blk[q++];
            if (nseq >= 128) {
                if (nseq < 255) {
                    if (q + 1 > bl) { status = ZSTDG_E_TRUNCATED; break; }
                    nseq = ((nseq - 128) << 8) + blk[q++];
                } else {
                    if (q + 2 > bl) { status = ZSTDG_E_TRUNCATED; break; }
                    nseq = blk[q] + (blk[q + 1] << 8) + 0x7F00;
                    q += 2;
                }
            }
            if (nseq == 0 && q != bl) { status = ZSTDG_E_CORRUPT; break; }
            int64_t lpos = 0;  // literals consumed
            BitB b;
            uint32_t sll = 0, sof = 0, sml = 0;
            if (nseq > 0) {
                if (lane == 0) {
                    int rc = 0;
                    do {
                        if (q >= bl) { rc = ZSTDG_E_TRUNCATED; break; }
                        const int modes = blk[q++];
                        if (modes & 3) { rc = ZSTDG_E_RESERVED; break; }
                        int u = seq_table(modes >> 6, blk + q, bl - q, S.ll, &ll_log, &have_ll, 9, 35, c_ll_def, 36, 6, S.norm);
                        if (u < 0) { rc = u; break; }
                        q += u;
                        u = seq_table((modes >> 4) & 3, blk + q, bl - q, S.of, &of_log, &have_of, 8, 31, c_of_def, 29, 5, S.norm);
                        if (u < 0) { rc = u; break; }
                        q += u;
                        u = seq_table((modes >> 2) & 3, blk + q, bl - q, S.ml, &ml_log, &have_ml, 9, 52, c_ml_def, 53, 6, S.norm);
                        if (u < 0) { rc = u; break; }
                        q += u;
                        if (b.init(blk + q, bl - q)) { rc = ZSTDG_E_CORRUPT; break; }
                        sll = b.read(ll_log);
                        sof = b.read(of_log);
                        sml = b.read(ml_log);
                    } while (0);
                    S.sh[0] = rc;
                }
                __syncwarp();
                status = S.sh[0];
                if (status) break;
            }
            int64_t out = produced;
            for (int s0 = 0; s0 < nseq && status == 0; s0 += ZSTDG_SEQ_BATCH) {
                const int cnt = min(ZSTDG_SEQ_BATCH, nseq - s0);
                if (lane == 0) {
                    int rc = 0;
                    for (int k = 0; k < cnt; k++) {
                        const uint32_t el = S.ll[sll], eo = S.of[sof], em = S.ml[sml];
                        const int lc = el & 0xff, oc = eo & 0xff, mc = em & 0xff;
                        if (oc > 31) { rc = ZSTDG_E_CORRUPT; break; }
                        uint32_t ofv = (1u << oc) + b.read(oc);
                        const uint32_t ml = c_ml_base[mc] + b.read(c_ml_bits[mc]);
                        const uint32_t ll = c_ll_base[lc] + b.read(c_ll_bits[lc]);
                        uint32_t off;
                        if (ofv > 3) {
                            off = ofv - 3;
                            rep[2] = rep[1]; rep[1] = rep[0]; rep[0] = off;
                        } else {
                            const int idx = (int)ofv - 1 + (ll == 0 ? 1 : 0);
                            if (idx == 0) off = rep[0];
                            else {
                                off = idx == 3 ? rep[0] - 1 : rep[idx];
                                if (off == 0) { rc = ZSTDG_E_OFFSET; break; }
                                if (idx != 1) rep[2] = rep[1];
                                rep[1] = rep[0];
                                rep[0] = off;
                            }
                        }
                        S.seq_ll[k] = ll; S.seq_ml[k] = ml; S.seq_of[k] = off;
                        if (s0 + k + 1 < nseq) {
                            sll = (el >> 16) + b.read((el >> 8) & 0xff);
                            sml = (em >> 16) + b.read((em >> 8) & 0xff);
                            sof = (eo >> 16) + b.read((eo >> 8) & 0xff);
                        }
                    }
                    if (!rc && s0 + cnt == nseq && b.pos != 0) rc = ZSTDG_E_CORRUPT;
                    S.sh[0] = rc;
                }
                __syncwarp();
                status = S.sh[0];
                if (status) break;
                // execute the batch
                for (int k = 0; k < cnt; k++) {
                    const int64_t ll = S.seq_ll[k], ml = S.seq_ml[k], off = S.seq_of[k];
                    if (lpos + ll > lit_n) { status = ZSTDG_E_CORRUPT; break; }
                    if (out + ll + ml > cap) { status = ZSTDG_E_DST_SIZE; break; }
                    if (off > out + ll || (window && (uint64_t)off > window)) { status = ZSTDG_E_OFFSET; break; }
                    // literals: read all, then write (the parked literals may lie just ahead of the write position)
                    for (int64_t j0 = 0; j0 < ll; j0 += 32) {
                        const int64_t j = j0 + lane;
                        uint8_t v = 0;
                        if (j < ll) v = ltype == 1 ? lit_rle : lit[lpos + j];
                        __syncwarp();
                        if (j < ll) dst[out + j] = v;
                    }
                    out += ll;
                    lpos += ll;
                    __syncwarp();
                    // match: byte j is out[j % off - off], produced before this copy
                    const uint8_t *from = dst + out - off;
                    const int64_t step = off > 32 ? 32 : 32 % off;
                    int64_t r = off > 32 ? lane : lane % off;
                    for (int64_t j0 = 0; j0 < ml; j0 += 32) {
                        if (j0 + lane < ml) dst[out + j0 + lane] = from[r];
                        r += step;
                        if (r >= off) r -= off;
                    }
                    out += ml;
                    __syncwarp();
                }
            }
            if (status) break;
            // the literals behind the last sequence
            const int64_t rest = lit_n - lpos;
            if (out + rest > cap) { status = ZSTDG_E_DST_SIZE; break; }
            for (int64_t j0 = 0; j0 < rest; j0 += 32) {
                const int64_t j = j0 + lane;
                uint8_t v = 0;
                if (j < rest) v = ltype == 1 ? lit_rle : lit[lpos + j];
                __syncwarp();
                if (j < rest) dst[out + j] = v;
            }
            out += rest;
            __syncwarp();
            if (out - produced > block_max) { status = ZSTDG_E_DST_SIZE; break; }
            produced = out;
        }
        if (status == 0 && content >= 0 && produced != content) status = ZSTDG_E_SIZE;
        if (status == 0 && checksum) {
            if (ip + 4 > slen) status = ZSTDG_E_TRUNCATED;
            else {
                const uint32_t want = (uint32_t)src[ip] | ((uint32_t)src[ip + 1] << 8) | ((uint32_t)src[ip + 2] << 16) | ((uint32_t)src[ip + 3] << 24);
                ip += 4;
                __syncwarp();
                const uint64_t h = xxh64_warp(dst, produced, lane);
                if ((uint32_t)h != want) status = ZSTDG_E_CHECKSUM;
            }
        }
        if (status == 0 && ip != slen) status = ZSTDG_E_TRAILING;
        if (lane == 0) {
            A.status[fi] = status ? status : (int32_t)produced;
            if (status && A.n_failed) atomicAdd(A.n_failed, 1);
        }
        __syncwarp();
    }
}

// Host screen of one read's bytes (no libzstd): 1 when they hold exactly one zstd frame that the device decodes --
// magic, no dictionary, a content size of at most `max_out` bytes, block headers walked to the last block, and the
// frame (plus its 4-byte checksum) spanning exactly `n` bytes.  *content receives the content size.  Anything else
// (skippable or concatenated frames, dictionaries, frames without a content size) stays on the host path.
static int zstd_screen(const uint8_t *p, size_t n, size_t max_out, uint64_t *content) {
    if (n < 6) return 0;
    const uint32_t magic = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    if (magic != 0xFD2FB528u) return 0;
    const int fhd = p[4], fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
    if ((fhd & 8) || did_flag != 0) return 0;
    const int fcs_sz = fcs_flag == 0 ? single : (1 << fcs_flag);
    if (fcs_sz == 0) return 0;
    size_t ip = 5 + (single ? 0 : 1);
    if (ip + fcs_sz > n) return 0;
    uint64_t v = 0;
    for (int k = 0; k < fcs_sz; k++) v |= (uint64_t)p[ip + k] << (8 * k);
    if (fcs_sz == 2) v += 256;
    ip += fcs_sz;
    if (v > max_out) return 0;
    for (;;) {
        if (ip + 3 > n) return 0;
        const uint32_t bh = (uint32_t)p[ip] | ((uint32_t)p[ip + 1] << 8) | ((uint32_t)p[ip + 2] << 16);
        const int type = (bh >> 1) & 3;
        if (type == 3) return 0;
        ip += 3 + (type == 1 ? 1 : (size_t)(bh >> 3));
        if (ip > n) return 0;
        if (bh & 1) break;
    }
    if (((fhd >> 2) & 1)) ip += 4;
    if (ip != n) return 0;
    *content = v;
    return 1;
}
