// Compressed ingest (SURVEY.md row f1): host entry points around svb16_decode_kernel.  Included at the end of
// adb_api.cu (uses its staging helpers).
#pragma once
#include "adb_svb16.cuh"
#include "adb_zstd.cuh"

// exclusive prefix sum of the samples per read -> element offsets of the decoded reads (int64 [n + 1]); one CTA
__global__ void __launch_bounds__(1024) svb_offsets_kernel(const int32_t *n_samples, int n, int64_t *offsets) {
    __shared__ long long wsum[32];
    __shared__ long long carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { carry = 0; offsets[0] = 0; }
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        long long v = (i < n) ? (long long)max(n_samples[i], 0) : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(ADB_FULL, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        long long wbase = 0;
        for (int w = 0; w < warp; w++) wbase += wsum[w];
        const long long c = carry;
        if (i < n) offsets[i + 1] = c + wbase + incl;
        __syncthreads();
        if (tid == 1023) carry = c + wbase + incl;
        __syncthreads();
    }
}

static int check_svb_batch(const adb_svb_batch *b) {
    if (!b || b->n_reads < 0 || b->m <= 0 || b->batch_size <= 0 ||
        (b->n_reads > 0 && (!b->comp || !b->comp_offsets || !b->n_samples || !b->full_lens || !b->calib_offset || !b->calib_scale))) {
        set_err("invalid adb_svb_batch");
        return ADB_ERR_ARG;
    }
    // one branch-free pass (it vectorizes): the pipelined calls run it before their first copy
    int outside = 0;
    for (int i = 0; i < b->n_reads; i++) outside |= (uint32_t)b->n_samples[i] > (uint32_t)b->m;
    if (outside) { set_err("n_samples outside [0, m]"); return ADB_ERR_ARG; }
    return ADB_OK;
}

// decode `nr` streams whose descriptors are already on the device (comp rebased so that comp[comp_off[i]] is valid)
static int launch_svb_decode(adb_ctx *ctx, const uint8_t *comp, const int64_t *comp_off, const int32_t *n_samples, int nr,
                             int64_t *offsets, int16_t *out, cudaStream_t st) {
    svb_offsets_kernel<<<1, 1024, 0, st>>>(n_samples, nr, offsets);
    SvbArgs A;
    A.comp = comp; A.comp_off = comp_off; A.n_samples = n_samples; A.out_off = offsets; A.out = out; A.n_reads = nr;
    const int warps_per_cta = ADB_SVB_THREADS / 32;
    const int grid = std::max(1, std::min((nr + warps_per_cta - 1) / warps_per_cta, ctx->sm_count * 8));
    {
        KernelTimer t(ctx, 6, st);
        svb16_decode_kernel<<<grid, ADB_SVB_THREADS, 0, st>>>(A);
    }
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

// decode `n` zstd frames whose descriptors are already on the device (src rebased so that src[src_off[i]] is valid);
// dst_cap nullptr: slot i ends at dst_off[i + 1]
static int launch_zstd_decode(adb_ctx *ctx, const uint8_t *src, const int64_t *src_off, uint8_t *dst, const int64_t *dst_off,
                              int32_t *status, int32_t *n_failed, int n, cudaStream_t st) {
    if (n <= 0) return ADB_OK;
    ZstdArgs A;
    A.src = src; A.src_off = src_off; A.dst = dst; A.dst_off = dst_off; A.dst_cap = nullptr; A.status = status;
    A.n_failed = n_failed; A.n = n;
    const int warps_per_cta = ZSTDG_THREADS / 32;
    const int grid = std::max(1, std::min((n + warps_per_cta - 1) / warps_per_cta, ctx->sm_count * 4));
    {
        KernelTimer t(ctx, 6, st);
        zstd_decode_kernel<<<grid, ZSTDG_THREADS, ZSTDG_SMEM, st>>>(A);
    }
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return ADB_OK;
}

extern "C" int adb_zstd_decompress_host(adb_ctx *ctx, const uint8_t *src, const int64_t *src_offsets, int32_t n, uint8_t *dst,
                                        const int64_t *dst_offsets, int32_t *status) {
    if (!ctx || n < 0 || (n > 0 && (!src || !src_offsets || !dst || !dst_offsets || !status))) { set_err("null argument"); return ADB_ERR_ARG; }
    if (n == 0) return ADB_OK;
    for (int i = 0; i < n; i++)
        if (src_offsets[i + 1] < src_offsets[i] || dst_offsets[i + 1] < dst_offsets[i]) { set_err("offsets must not decrease"); return ADB_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StreamDrain drain;
    drain.add(st);
    ChunkBufs &b = ctx->p[0];
    const int64_t s0 = src_offsets[0], d0 = dst_offsets[0];
    const size_t sbytes = (size_t)(src_offsets[n] - s0), dbytes = (size_t)(dst_offsets[n] - d0);
    if (b.frames.ensure(sbytes + 16) || b.foffs.ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        b.comp.ensure(dbytes + 16) || b.coffs.ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        b.zstat.ensure(sizeof(int32_t) * (size_t)n + 16)) { set_err("cudaMalloc zstd staging"); return ADB_ERR_CUDA; }
    if (sbytes) CUDA_TRY(cudaMemcpyAsync(b.frames.p, src + s0, sbytes, cudaMemcpyHostToDevice, st));
    // the slots start as the caller left them: bytes the decoder does not write come back unchanged
    if (dbytes) CUDA_TRY(cudaMemcpyAsync(b.comp.p, dst + d0, dbytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b.foffs.p, src_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b.coffs.p, dst_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    int rc = launch_zstd_decode(ctx, (const uint8_t *)b.frames.p - s0, (const int64_t *)b.foffs.p,
                                (uint8_t *)b.comp.p - d0, (const int64_t *)b.coffs.p, (int32_t *)b.zstat.p,
                                nullptr, n, st);
    if (rc) return rc;
    if (dbytes) CUDA_TRY(cudaMemcpyAsync(dst + d0, b.comp.p, dbytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(status, b.zstat.p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    drain.armed = false;
    return ADB_OK;
}

extern "C" int adb_svb16_decode_host(adb_ctx *ctx, const adb_svb_batch *batch, int16_t *out_adc) {
    if (!ctx || !out_adc) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_svb_batch(batch);
    if (rc) return rc;
    const int n = batch->n_reads;
    if (n == 0) return ADB_OK;
    int64_t total = 0;
    for (int i = 0; i < n; i++) total += batch->n_samples[i];
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StreamDrain drain;
    drain.add(st);
    ChunkBufs &b = ctx->p[0];
    const int64_t c0 = batch->comp_offsets[0], c1 = batch->comp_offsets[n];
    const size_t cbytes = (size_t)(c1 - c0) + 16;
    if (b.comp.ensure(cbytes + 64) || b.coffs.ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        b.nsamp.ensure(sizeof(int32_t) * (size_t)n + 16) || b.offsets.ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        b.signal.ensure((size_t)total * 2 + 64)) { set_err("cudaMalloc svb16 staging"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(b.comp.p, batch->comp + c0, cbytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b.coffs.p, batch->comp_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b.nsamp.p, batch->n_samples, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    rc = launch_svb_decode(ctx, (const uint8_t *)b.comp.p - c0, (const int64_t *)b.coffs.p,
                           (const int32_t *)b.nsamp.p, n, (int64_t *)b.offsets.p, (int16_t *)b.signal.p, st);
    if (rc) return rc;
    if (total > 0) CUDA_TRY(cudaMemcpyAsync(out_adc, b.signal.p, (size_t)total * 2, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    drain.armed = false;
    return ADB_OK;
}

// chunk schedule of the pipelined entry points (in minibatches): small chunks at both ends (the first copy and the
// last chunk's kernels overlap nothing), full-size chunks in between
static std::vector<int> pipeline_schedule(int n_batches, int chunk_batches) {
    std::vector<int> sched, tail;
    const int q = std::max(1, chunk_batches / 4), h = std::max(1, chunk_batches / 2);
    int left = n_batches;
    if (n_batches >= 2 * (q + h) + chunk_batches) {
        sched.push_back(q); sched.push_back(h);
        tail.push_back(h); tail.push_back(q);
        left -= 2 * (q + h);
    }
    while (left > 0) { const int c = std::min(left, chunk_batches); sched.push_back(c); left -= c; }
    sched.insert(sched.end(), tail.begin(), tail.end());
    return sched;
}

// Before the first chunk of a pipelined call: create the twin when `want_twin` asks for it (consecutive chunks
// alternate between ctx and its twin: own compute stream, own scratch), give the twin the options of ctx, and upload
// the CNN weights to every context in use.  Without a twin, cc[1] and w_devs[1] repeat cc[0] and w_devs[0].
static int pair_setup(adb_ctx *ctx, bool want_twin, const adb_config *cfg, const float *cnn_weights, adb_ctx *cc[2],
                      const float *w_devs[2]) {
    if (cfg->primary_method == ADB_METHOD_CNN && !cnn_weights) { set_err("cnn_weights required"); return ADB_ERR_ARG; }
    if (want_twin && !ctx->twin) {
        int rc = adb_ctx_create(ctx->device, &ctx->twin);
        if (rc) return rc;
    }
    if (ctx->twin) ctx->twin->opt = ctx->opt;
    cc[0] = ctx;
    cc[1] = ctx->twin ? ctx->twin : ctx;
    w_devs[0] = w_devs[1] = nullptr;
    if (cfg->primary_method != ADB_METHOD_CNN) return ADB_OK;
    for (int k = 0; k < (ctx->twin ? 2 : 1); k++) {
        int rc = upload_cnn_weights(cc[k], cnn_weights, &w_devs[k]);
        if (rc) return rc;
    }
    if (!ctx->twin) w_devs[1] = w_devs[0];
    return ADB_OK;
}

enum { CHUNK_RAW = 0, CHUNK_SVB16 = 1, CHUNK_ZSTD = 2 };

// One chunk of reads in host memory.  The offsets may index a larger buffer: the chunk's payload starts at offsets[0]
// (dec_offsets[0] for the decoded streams), and the staged copies are addressed through pointers rebased by it.
struct ChunkDesc {
    int rep = CHUNK_RAW;  // raw int16 samples, svb16 streams, or one zstd frame per read over its svb16 stream
    const void *payload = nullptr;
    size_t payload_bytes = 0;              // svb16: with the 16 bytes of slack behind the last stream
    const int64_t *offsets = nullptr;      // [nr + 1] samples (raw), streams (svb16) or frames (zstd)
    const int64_t *dec_offsets = nullptr;  // zstd: [nr + 1] 16-byte aligned slots of the decoded svb16 streams
    const int32_t *n_samples = nullptr;    // [nr] samples per read; raw chunks may leave it null
    const int32_t *full_lens = nullptr;
    const float *calib_offset = nullptr, *calib_scale = nullptr;
    int nr = 0, nb = 0, m = 0, batch_size = 0;
};

// Stages chunk k in slot `slot` of context c and enqueues all of its work.  The H2D copies go on the copy stream cs;
// on c's stream follow the zstd decode (refused frames counted in z_fail) and the svb16 decode that k.rep needs,
// detection (skipped when !run), and the D2H copies of the records and, when out_status is given, the minibatch status.
static int enqueue_chunk(adb_ctx *c, int slot, cudaStream_t cs, const ChunkDesc &k, const adb_config *cfg, const float *w_dev,
                         int32_t *z_fail, bool run, adb_record *out_records, int32_t *out_status) {
    ChunkBufs &b = c->p[slot];
    const cudaStream_t ks = c->stream;
    const int nr = k.nr;
    const size_t n8 = sizeof(int64_t) * ((size_t)nr + 1), n4 = sizeof(int32_t) * (size_t)nr;
    // the decoded reads: the raw payload, or n_samples in total (counted while the slot's previous chunk still runs)
    size_t sig_bytes = k.payload_bytes;
    if (k.rep != CHUNK_RAW) {
        int64_t samples = 0;
        for (int i = 0; i < nr; i++) samples += k.n_samples[i];
        sig_bytes = 2 * (size_t)samples;
    }
    // the slot is free once the chunk that used it last has been copied back
    CUDA_TRY(cudaEventSynchronize(b.done));
    const int64_t dec0 = k.rep == CHUNK_ZSTD ? k.dec_offsets[0] : 0, dec_bytes = k.rep == CHUNK_ZSTD ? k.dec_offsets[nr] - dec0 : 0;
    DevBuf &in = k.rep == CHUNK_ZSTD ? b.frames : k.rep == CHUNK_SVB16 ? b.comp : b.signal;
    DevBuf &in_off = k.rep == CHUNK_ZSTD ? b.foffs : k.rep == CHUNK_SVB16 ? b.coffs : b.offsets;
    if (b.signal.ensure(sig_bytes + 64) || b.offsets.ensure(n8) || b.lens.ensure(n4 + 16) || b.coff.ensure(n4 + 16) ||
        b.cscale.ensure(n4 + 16) || b.records.ensure(sizeof(adb_record) * (size_t)nr) || b.status.ensure(sizeof(int) * (size_t)k.nb + 16) ||
        (k.n_samples && b.nsamp.ensure(n4 + 16)) ||
        (k.rep != CHUNK_RAW && (b.coffs.ensure(n8) || b.comp.ensure((k.rep == CHUNK_ZSTD ? (size_t)dec_bytes : k.payload_bytes) + 64))) ||
        (k.rep == CHUNK_ZSTD && (b.frames.ensure(k.payload_bytes + 16) || b.foffs.ensure(n8) || b.zstat.ensure(n4 + 16)))) {
        set_err("cudaMalloc pipeline staging");
        return ADB_ERR_CUDA;
    }
    CUDA_TRY(cudaMemcpyAsync(in.p, k.payload, k.payload_bytes, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(in_off.p, k.offsets, n8, cudaMemcpyHostToDevice, cs));
    if (k.rep == CHUNK_ZSTD) CUDA_TRY(cudaMemcpyAsync(b.coffs.p, k.dec_offsets, n8, cudaMemcpyHostToDevice, cs));
    if (k.n_samples) CUDA_TRY(cudaMemcpyAsync(b.nsamp.p, k.n_samples, n4, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(b.lens.p, k.full_lens, n4, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(b.coff.p, k.calib_offset, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaMemcpyAsync(b.cscale.p, k.calib_scale, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaEventRecord(b.copied, cs));
    CUDA_TRY(cudaStreamWaitEvent(ks, b.copied, 0));
    if (run) {
        const int64_t base = k.offsets[0];
        const int16_t *signal = (const int16_t *)b.signal.p;
        int rc = ADB_OK;
        if (k.rep == CHUNK_RAW) {
            signal -= base;  // the offsets stay as given
        } else {
            const uint8_t *streams = (const uint8_t *)b.comp.p - base;
            if (k.rep == CHUNK_ZSTD) {
                uint8_t *dec = (uint8_t *)b.comp.p - dec0;
                CUDA_TRY(cudaMemsetAsync((uint8_t *)b.comp.p + dec_bytes, 0, 16, ks));  // the slack behind the last stream
                rc = launch_zstd_decode(c, (const uint8_t *)b.frames.p - base, (const int64_t *)b.foffs.p, dec,
                                        (const int64_t *)b.coffs.p, (int32_t *)b.zstat.p, z_fail, nr, ks);
                if (rc) return rc;
                streams = dec;
            }
            rc = launch_svb_decode(c, streams, (const int64_t *)b.coffs.p, (const int32_t *)b.nsamp.p, nr, (int64_t *)b.offsets.p,
                                   (int16_t *)b.signal.p, ks);
            if (rc) return rc;
        }
        adb_batch d;
        d.signal = signal; d.sig_type = ADB_SIG_I16; d.n_reads = nr; d.m = k.m; d.batch_size = k.batch_size;
        d.offsets = (const int64_t *)b.offsets.p; d.full_lens = (const int32_t *)b.lens.p;
        d.calib_offset = (const float *)b.coff.p; d.calib_scale = (const float *)b.cscale.p;
        rc = adb_detect_dev(c, &d, cfg, w_dev, (adb_record *)b.records.p, (int *)b.status.p, ks);
        if (rc) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(out_records, b.records.p, sizeof(adb_record) * (size_t)nr, cudaMemcpyDeviceToHost, ks));
    if (out_status) CUDA_TRY(cudaMemcpyAsync(out_status, b.status.p, sizeof(int) * (size_t)k.nb, cudaMemcpyDeviceToHost, ks));
    CUDA_TRY(cudaEventRecord(b.done, ks));
    return ADB_OK;
}

// The chunk loop of the pipelined host entry points.  Reads [r0, r1) of each scheduled chunk go through enqueue_chunk;
// set_payload(k, r0, r1) fills in what depends on the input form.  All copies go through ctx's copy stream in order;
// with a twin, every chunk of a context uses its slot 0, otherwise consecutive chunks alternate between ctx's slots.
template <class Batch, class SetPayload>
static int detect_pipelined(adb_ctx *ctx, const Batch &batch, const adb_config *cfg, const float *cnn_weights,
                            adb_record *out_records, int32_t *batch_status, int32_t chunk_batches, int32_t *z_fail,
                            SetPayload set_payload) {
    const int bs = batch.batch_size;
    const std::vector<int> sched = pipeline_schedule((batch.n_reads + bs - 1) / bs, std::max(1, chunk_batches));
    adb_ctx *cc[2];
    const float *w_devs[2];
    int rc = pair_setup(ctx, sched.size() >= 3, cfg, cnn_weights, cc, w_devs);
    if (rc) return rc;
    cudaStream_t cs = ctx->copy_stream;
    StreamDrain drain;
    drain.add(cs);
    drain.add(ctx->stream);
    if (ctx->twin) drain.add(ctx->twin->stream);
    for (int ch = 0, b0 = 0; ch < (int)sched.size(); b0 += sched[ch++]) {
        const int r0 = b0 * bs, r1 = (int)std::min<long long>((long long)batch.n_reads, (long long)(b0 + sched[ch]) * bs);
        ChunkDesc k;
        k.nr = r1 - r0;
        k.nb = (k.nr + bs - 1) / bs;
        k.m = batch.m;
        k.batch_size = bs;
        k.full_lens = batch.full_lens + r0;
        k.calib_offset = batch.calib_offset + r0;
        k.calib_scale = batch.calib_scale + r0;
        set_payload(k, r0, r1);
        rc = enqueue_chunk(cc[ch & 1], ctx->twin ? 0 : (ch & 1), cs, k, cfg, w_devs[ch & 1], z_fail, !ctx->opt.copy_only,
                           out_records + r0, batch_status ? batch_status + b0 : nullptr);
        if (rc) return rc;
    }
    if (ctx->twin) CUDA_TRY(cudaStreamSynchronize(ctx->twin->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(cs));
    drain.armed = false;
    return ADB_OK;
}

// Pipelined ingest for long jobs: the reads are cut into chunks of `chunk_batches` minibatches; the H2D copy of
// chunk i+1 (copy stream) overlaps the kernels of chunk i (compute stream), records return per chunk.  Host buffers
// should be pinned (cudaHostAlloc / torch pin_memory) for the copies to be asynchronous.  I16 ragged input only.
extern "C" int adb_detect_pipelined_host(adb_ctx *ctx, const adb_batch *batch, const adb_config *cfg,
                                         const float *cnn_weights, adb_record *out_records, int32_t *batch_status,
                                         int32_t chunk_batches) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    if (batch->sig_type != ADB_SIG_I16) { set_err("pipelined ingest takes ragged int16 input"); return ADB_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (batch->n_reads == 0) return ADB_OK;
    return detect_pipelined(ctx, *batch, cfg, cnn_weights, out_records, batch_status, chunk_batches, nullptr,
                            [&](ChunkDesc &k, int r0, int r1) {
                                k.payload = (const int16_t *)batch->signal + batch->offsets[r0];
                                k.payload_bytes = (size_t)(batch->offsets[r1] - batch->offsets[r0]) * 2;
                                k.offsets = batch->offsets + r0;
                            });
}

// adb_detect_pipelined_svb_host (vbz = false) and adb_detect_pipelined_vbz_host (vbz = true: batch->comp holds one
// zstd frame per read, decoded on the device into the svb16 layout before svb16_decode_kernel)
static int detect_pipelined_comp(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                                 adb_record *out_records, int32_t *batch_status, int32_t chunk_batches, bool vbz) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_svb_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (batch->n_reads == 0) return ADB_OK;
    // VBZ: every frame is screened on the host (content size -> layout of the decoded streams: 16-byte aligned, 16 bytes
    // of slack behind the last one); a frame the device does not take is refused here
    std::vector<int64_t> dec_off;
    if (vbz) {
        const size_t per_read_cap = (size_t)batch->m * 2 + (size_t)((batch->m + 7) / 8 + 3) + 32;
        dec_off.resize((size_t)batch->n_reads + 1);
        dec_off[0] = 0;
        for (int i = 0; i < batch->n_reads; i++) {
            const int64_t o0 = batch->comp_offsets[i], o1 = batch->comp_offsets[i + 1];
            uint64_t cs = 0;
            if (o1 < o0 || !zstd_screen(batch->comp + o0, (size_t)(o1 - o0), per_read_cap, &cs)) {
                set_err("read " + std::to_string(i) + ": not one zstd frame with a content size and no dictionary");
                return ADB_ERR_UNSUPPORTED;
            }
            dec_off[i + 1] = dec_off[i] + (int64_t)((cs + 15) & ~(uint64_t)15);
        }
        // one counter for the call and both contexts, cleared on the copy stream: every chunk's kernels wait for its copies
        if (ctx->z_fail.ensure(16)) { set_err("cudaMalloc zstd counter"); return ADB_ERR_CUDA; }
        CUDA_TRY(cudaMemsetAsync(ctx->z_fail.p, 0, sizeof(int32_t), ctx->copy_stream));
    }
    rc = detect_pipelined(ctx, *batch, cfg, cnn_weights, out_records, batch_status, chunk_batches,
                          vbz ? (int32_t *)ctx->z_fail.p : nullptr, [&](ChunkDesc &k, int r0, int r1) {
                              const int64_t c0 = batch->comp_offsets[r0], c1 = batch->comp_offsets[r1];
                              k.rep = vbz ? CHUNK_ZSTD : CHUNK_SVB16;
                              k.payload = batch->comp + c0;
                              k.payload_bytes = (size_t)(c1 - c0) + (vbz ? 0 : 16);  // svb16: the slack travels along
                              k.offsets = batch->comp_offsets + r0;
                              k.dec_offsets = vbz ? dec_off.data() + r0 : nullptr;
                              k.n_samples = batch->n_samples + r0;
                          });
    if (rc) return rc;
    if (vbz && !ctx->opt.copy_only) {
        int32_t n_failed = 0;
        CUDA_TRY(cudaMemcpy(&n_failed, ctx->z_fail.p, sizeof(int32_t), cudaMemcpyDeviceToHost));
        if (n_failed) {
            set_err(std::to_string(n_failed) + " zstd frame(s) do not decompress to their stated size");
            return ADB_ERR_ARG;
        }
    }
    return ADB_OK;
}

extern "C" int adb_detect_pipelined_svb_host(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg,
                                             const float *cnn_weights, adb_record *out_records, int32_t *batch_status,
                                             int32_t chunk_batches) {
    return detect_pipelined_comp(ctx, batch, cfg, cnn_weights, out_records, batch_status, chunk_batches, false);
}

extern "C" int adb_detect_pipelined_vbz_host(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg,
                                             const float *cnn_weights, adb_record *out_records, int32_t *batch_status,
                                             int32_t chunk_batches) {
    return detect_pipelined_comp(ctx, batch, cfg, cnn_weights, out_records, batch_status, chunk_batches, true);
}
