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
    const int64_t s0 = src_offsets[0], d0 = dst_offsets[0];
    const size_t sbytes = (size_t)(src_offsets[n] - s0), dbytes = (size_t)(dst_offsets[n] - d0);
    if (ctx->p_frames[0].ensure(sbytes + 16) || ctx->p_foffs[0].ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        ctx->p_comp[0].ensure(dbytes + 16) || ctx->p_coffs[0].ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        ctx->p_zstat[0].ensure(sizeof(int32_t) * (size_t)n + 16)) { set_err("cudaMalloc zstd staging"); return ADB_ERR_CUDA; }
    if (sbytes) CUDA_TRY(cudaMemcpyAsync(ctx->p_frames[0].p, src + s0, sbytes, cudaMemcpyHostToDevice, st));
    // the slots start as the caller left them: bytes the decoder does not write come back unchanged
    if (dbytes) CUDA_TRY(cudaMemcpyAsync(ctx->p_comp[0].p, dst + d0, dbytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->p_foffs[0].p, src_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->p_coffs[0].p, dst_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    int rc = launch_zstd_decode(ctx, (const uint8_t *)ctx->p_frames[0].p - s0, (const int64_t *)ctx->p_foffs[0].p,
                                (uint8_t *)ctx->p_comp[0].p - d0, (const int64_t *)ctx->p_coffs[0].p, (int32_t *)ctx->p_zstat[0].p,
                                nullptr, n, st);
    if (rc) return rc;
    if (dbytes) CUDA_TRY(cudaMemcpyAsync(dst + d0, ctx->p_comp[0].p, dbytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(status, ctx->p_zstat[0].p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
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
    for (int i = 0; i < n; i++) {
        if (batch->n_samples[i] < 0 || batch->n_samples[i] > batch->m) { set_err("n_samples outside [0, m]"); return ADB_ERR_ARG; }
        total += batch->n_samples[i];
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    StreamDrain drain;
    drain.add(st);
    const int64_t c0 = batch->comp_offsets[0], c1 = batch->comp_offsets[n];
    const size_t cbytes = (size_t)(c1 - c0) + 16;
    if (ctx->p_comp[0].ensure(cbytes + 64) || ctx->p_coffs[0].ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        ctx->p_nsamp[0].ensure(sizeof(int32_t) * (size_t)n + 16) || ctx->p_offsets[0].ensure(sizeof(int64_t) * ((size_t)n + 1)) ||
        ctx->p_signal[0].ensure((size_t)total * 2 + 64)) { set_err("cudaMalloc svb16 staging"); return ADB_ERR_CUDA; }
    CUDA_TRY(cudaMemcpyAsync(ctx->p_comp[0].p, batch->comp + c0, cbytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->p_coffs[0].p, batch->comp_offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->p_nsamp[0].p, batch->n_samples, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    rc = launch_svb_decode(ctx, (const uint8_t *)ctx->p_comp[0].p - c0, (const int64_t *)ctx->p_coffs[0].p,
                           (const int32_t *)ctx->p_nsamp[0].p, n, (int64_t *)ctx->p_offsets[0].p, (int16_t *)ctx->p_signal[0].p, st);
    if (rc) return rc;
    if (total > 0) CUDA_TRY(cudaMemcpyAsync(out_adc, ctx->p_signal[0].p, (size_t)total * 2, cudaMemcpyDeviceToHost, st));
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

// adb_detect_pipelined_svb_host (vbz = false) and adb_detect_pipelined_vbz_host (vbz = true: batch->comp holds one
// zstd frame per read, decoded on the device into the svb16 layout before svb16_decode_kernel)
static int detect_pipelined_comp(adb_ctx *ctx, const adb_svb_batch *batch, const adb_config *cfg, const float *cnn_weights,
                                 adb_record *out_records, int32_t *batch_status, int32_t chunk_batches, bool vbz) {
    if (!ctx || !out_records) { set_err("null argument"); return ADB_ERR_ARG; }
    int rc = check_svb_batch(batch);
    if (rc) return rc;
    rc = check_config(cfg);
    if (rc) return rc;
    if (chunk_batches < 1) chunk_batches = 1;
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
    }
    if (vbz && ctx->z_fail.ensure(16)) { set_err("cudaMalloc zstd counter"); return ADB_ERR_CUDA; }
    // (on the copy stream: every chunk's kernels wait for its copies)
    if (vbz) CUDA_TRY(cudaMemsetAsync(ctx->z_fail.p, 0, sizeof(int32_t), ctx->copy_stream));
    const int n_batches = (batch->n_reads + batch->batch_size - 1) / batch->batch_size;
    const std::vector<int> sched = pipeline_schedule(n_batches, chunk_batches);
    if (!ctx->twin && sched.size() >= 3) {
        rc = adb_ctx_create(ctx->device, &ctx->twin);
        if (rc) return rc;
    }
    if (ctx->twin) {
        ctx->twin->opt_no_fast_validate = ctx->opt_no_fast_validate;
        ctx->twin->opt_hist_validate = ctx->opt_hist_validate;
        ctx->twin->opt_cnn_fp32 = ctx->opt_cnn_fp32;
        ctx->twin->opt_exact_gsel = ctx->opt_exact_gsel;
        ctx->twin->opt_no_cand_followup = ctx->opt_no_cand_followup;
    }
    adb_ctx *cc[2] = {ctx, ctx->twin ? ctx->twin : ctx};
    const float *w_devs[2] = {nullptr, nullptr};
    if (cfg->primary_method == ADB_METHOD_CNN) {
        if (!cnn_weights) { set_err("cnn_weights required"); return ADB_ERR_ARG; }
        for (int k = 0; k < (ctx->twin ? 2 : 1); k++) {
            if (cc[k]->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc weights"); return ADB_ERR_CUDA; }
            CUDA_TRY(cudaMemcpyAsync(cc[k]->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, cc[k]->stream));
            w_devs[k] = (const float *)cc[k]->h_misc2.p;
        }
        if (!ctx->twin) w_devs[1] = w_devs[0];
    }
    cudaStream_t cs = ctx->copy_stream;
    StreamDrain drain;
    drain.add(cs);
    drain.add(ctx->stream);
    if (ctx->twin) drain.add(ctx->twin->stream);
    int b0 = 0;
    for (int ch = 0; ch < (int)sched.size(); ch++) {
        adb_ctx *c = cc[ch & 1];
        const int slot = ctx->twin ? 0 : (ch & 1);
        cudaStream_t ks = c->stream;
        const int r0 = b0 * batch->batch_size;
        const int r1 = (int)std::min<long long>((long long)batch->n_reads, (long long)(b0 + sched[ch]) * batch->batch_size), nr = r1 - r0;
        const int nb = (nr + batch->batch_size - 1) / batch->batch_size;
        const int64_t c0 = batch->comp_offsets[r0], c1 = batch->comp_offsets[r1];
        const size_t cbytes = (size_t)(c1 - c0) + 16;  // the slack behind the last stream travels along
        // the decoded reads of the chunk: at most nr * m samples; the exact size follows from the compressed size
        // (a stream holds at least one byte per sample)
        const size_t dec_cap = std::min<size_t>((size_t)nr * (size_t)batch->m, (size_t)(c1 - c0));
        if (ch >= 2) CUDA_TRY(cudaEventSynchronize(c->p_done[slot]));
        if (c->p_comp[slot].ensure(cbytes + 64) || c->p_coffs[slot].ensure(sizeof(int64_t) * ((size_t)nr + 1)) ||
            c->p_nsamp[slot].ensure(sizeof(int32_t) * (size_t)nr + 16) || c->p_signal[slot].ensure(dec_cap * 2 + 64) ||
            c->p_offsets[slot].ensure(sizeof(int64_t) * ((size_t)nr + 1)) || c->p_lens[slot].ensure(sizeof(int32_t) * (size_t)nr + 16) ||
            c->p_coff[slot].ensure(sizeof(float) * (size_t)nr + 16) || c->p_cscale[slot].ensure(sizeof(float) * (size_t)nr + 16) ||
            c->p_records[slot].ensure(sizeof(adb_record) * (size_t)nr) || c->p_status[slot].ensure(sizeof(int) * (size_t)nb + 16)) {
            set_err("cudaMalloc pipeline staging");
            return ADB_ERR_CUDA;
        }
        if (vbz) {  // frames travel; the decoded streams are laid out from dec_off rebased to the chunk
            const int64_t d0 = dec_off[r0], dbytes = dec_off[r1] - d0;
            if (c->p_frames[slot].ensure((size_t)(c1 - c0) + 16) || c->p_foffs[slot].ensure(sizeof(int64_t) * ((size_t)nr + 1)) ||
                c->p_comp[slot].ensure((size_t)dbytes + 64) || c->p_zstat[slot].ensure(sizeof(int32_t) * (size_t)nr + 16) ||
                c->p_signal[slot].ensure(std::min<size_t>((size_t)nr * (size_t)batch->m, (size_t)dbytes) * 2 + 64)) {
                set_err("cudaMalloc pipeline staging");
                return ADB_ERR_CUDA;
            }
            CUDA_TRY(cudaMemcpyAsync(c->p_frames[slot].p, batch->comp + c0, (size_t)(c1 - c0), cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(c->p_foffs[slot].p, batch->comp_offsets + r0, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(c->p_coffs[slot].p, dec_off.data() + r0, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
        } else {
            CUDA_TRY(cudaMemcpyAsync(c->p_comp[slot].p, batch->comp + c0, cbytes, cudaMemcpyHostToDevice, cs));
            CUDA_TRY(cudaMemcpyAsync(c->p_coffs[slot].p, batch->comp_offsets + r0, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
        }
        CUDA_TRY(cudaMemcpyAsync(c->p_nsamp[slot].p, batch->n_samples + r0, sizeof(int32_t) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_lens[slot].p, batch->full_lens + r0, sizeof(int32_t) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_coff[slot].p, batch->calib_offset + r0, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaMemcpyAsync(c->p_cscale[slot].p, batch->calib_scale + r0, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaEventRecord(c->p_copied[slot], cs));
        CUDA_TRY(cudaStreamWaitEvent(ks, c->p_copied[slot], 0));
        if (!ctx->opt_copy_only) {
            int64_t sbase = c0;
            if (vbz) {
                sbase = dec_off[r0];
                uint8_t *dec = (uint8_t *)c->p_comp[slot].p - sbase;
                CUDA_TRY(cudaMemsetAsync(dec + dec_off[r1], 0, 16, ks));
                rc = launch_zstd_decode(c, (const uint8_t *)c->p_frames[slot].p - c0, (const int64_t *)c->p_foffs[slot].p, dec,
                                        (const int64_t *)c->p_coffs[slot].p, (int32_t *)c->p_zstat[slot].p, (int32_t *)ctx->z_fail.p, nr, ks);
                if (rc) return rc;
            }
            rc = launch_svb_decode(c, (const uint8_t *)c->p_comp[slot].p - sbase, (const int64_t *)c->p_coffs[slot].p,
                                   (const int32_t *)c->p_nsamp[slot].p, nr, (int64_t *)c->p_offsets[slot].p,
                                   (int16_t *)c->p_signal[slot].p, ks);
            if (rc) return rc;
            adb_batch d;
            d.signal = c->p_signal[slot].p;
            d.sig_type = ADB_SIG_I16;
            d.n_reads = nr;
            d.m = batch->m;
            d.batch_size = batch->batch_size;
            d.offsets = (const int64_t *)c->p_offsets[slot].p;
            d.full_lens = (const int32_t *)c->p_lens[slot].p;
            d.calib_offset = (const float *)c->p_coff[slot].p;
            d.calib_scale = (const float *)c->p_cscale[slot].p;
            rc = adb_detect_dev(c, &d, cfg, w_devs[ch & 1], (adb_record *)c->p_records[slot].p, (int *)c->p_status[slot].p, ks);
            if (rc) return rc;
        }
        CUDA_TRY(cudaMemcpyAsync(out_records + r0, c->p_records[slot].p, sizeof(adb_record) * (size_t)nr, cudaMemcpyDeviceToHost, ks));
        if (batch_status)
            CUDA_TRY(cudaMemcpyAsync(batch_status + b0, c->p_status[slot].p, sizeof(int) * (size_t)nb, cudaMemcpyDeviceToHost, ks));
        CUDA_TRY(cudaEventRecord(c->p_done[slot], ks));
        b0 += sched[ch];
    }
    if (ctx->twin) CUDA_TRY(cudaStreamSynchronize(ctx->twin->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(cs));
    drain.armed = false;
    if (vbz && !ctx->opt_copy_only) {
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
