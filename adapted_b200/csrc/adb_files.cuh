// Native file-level pipeline (SURVEY.md row f1): signal containers -> GPU detection -> boundary tables, every stage
// overlapped.  Replaces, for one GPU, the producer thread (adapted/file_proc.py:143-214), the process pool
// (:738-784), the two saver threads (:312-457) and run_detect's bookkeeping (:612-823).
//
//   reader thread     walks the files in order, cuts the selected reads into chunks of `chunk_batches` minibatches
//                     (minibatches run across file boundaries like the reference's generator) and fills a ring of
//                     PINNED host slots: the reads' compressed streams are copied (several copy threads per chunk) or,
//                     for zstd containers (pod5's VBZ = zstd over svb16), decompressed straight into the slot
//   GPU thread        (the caller) per slot: async H2D of the compressed chunk on the copy stream, svb16 decode +
//                     detection on the compute stream of alternating contexts, async D2H of the records into the slot
//   writer thread     waits for a slot's records, splits them into the pass / fail lists in arrival order and hands
//                     every full table (batch_size_output reads) to
//   formatter threads adb_format_csv_ex + one write() per table: detected_boundaries_<i>.csv / failed_reads_<i>.csv
//
// Container "ADBSIG02" (adapted_b200/ingest.py writes it): a 128-byte header, then 64-byte aligned sections.
// Included at the end of adb_api.cu.
#pragma once
#include <sched.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <thread>

#include "adb_ingest.cuh"

namespace adbf {

// CPUs this process may run on (a rank of a multi-GPU job is bound to its GPU's PCIe-local set: bench.py)
static unsigned usable_cpus() {
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0) { const int n = CPU_COUNT(&set); if (n > 0) return (unsigned)n; }
    return std::max(1u, std::thread::hardware_concurrency());
}

#pragma pack(push, 1)
struct Header {
    char magic[8];
    uint32_t version, flags;
    uint64_t n_reads;
    uint32_t id_width, reserved0;
    uint64_t off_comp_offsets, off_n_samples, off_full_lens, off_calib_offset, off_calib_scale, off_read_ids, off_blob, blob_bytes;
    uint8_t reserved[32];
};
#pragma pack(pop)
static_assert(sizeof(Header) == 128, "container header is 128 bytes");

enum { F_SVB16 = 1, F_ZSTD = 2 };
static const int ID_SLOT_WIDTH = 64;

struct SigFile {
    int fd = -1;
    size_t size = 0;
    const uint8_t *base = nullptr;
    Header h;
    const int64_t *coffs = nullptr;
    const int32_t *nsamp = nullptr, *lens = nullptr;
    const float *coff = nullptr, *cscale = nullptr;
    const char *ids = nullptr;
    const uint8_t *blob = nullptr;
    void close_() {
        if (base) munmap((void *)base, size);
        if (fd >= 0) close(fd);
        base = nullptr;
        fd = -1;
    }
};

static int open_sigfile(const char *path, SigFile &f) {
    f.fd = open(path, O_RDONLY);
    if (f.fd < 0) { set_err(std::string("cannot open ") + path); return ADB_ERR_ARG; }
    struct stat st;
    if (fstat(f.fd, &st) != 0 || (size_t)st.st_size < sizeof(Header)) { set_err(std::string("not a signal container: ") + path); f.close_(); return ADB_ERR_ARG; }
    f.size = (size_t)st.st_size;
    f.base = (const uint8_t *)mmap(nullptr, f.size, PROT_READ, MAP_SHARED, f.fd, 0);
    if (f.base == MAP_FAILED) { f.base = nullptr; set_err(std::string("mmap failed: ") + path); f.close_(); return ADB_ERR_ARG; }
    memcpy(&f.h, f.base, sizeof(Header));
    const Header &h = f.h;
    const uint64_t n = h.n_reads;
    auto inside = [&](uint64_t off, uint64_t bytes) { return off <= f.size && bytes <= f.size - off; };
    if (memcmp(h.magic, "ADBSIG02", 8) != 0 || h.version != 2 || n > 0x7fffffffull || h.id_width == 0 || h.id_width > ID_SLOT_WIDTH ||
        !inside(h.off_comp_offsets, 8 * (n + 1)) || !inside(h.off_n_samples, 4 * n) || !inside(h.off_full_lens, 4 * n) ||
        !inside(h.off_calib_offset, 4 * n) || !inside(h.off_calib_scale, 4 * n) || !inside(h.off_read_ids, (uint64_t)h.id_width * n) ||
        !inside(h.off_blob, h.blob_bytes)) {
        set_err(std::string("not an ADBSIG02 signal container (or truncated): ") + path);
        f.close_();
        return ADB_ERR_ARG;
    }
    f.coffs = (const int64_t *)(f.base + h.off_comp_offsets);
    f.nsamp = (const int32_t *)(f.base + h.off_n_samples);
    f.lens = (const int32_t *)(f.base + h.off_full_lens);
    f.coff = (const float *)(f.base + h.off_calib_offset);
    f.cscale = (const float *)(f.base + h.off_calib_scale);
    f.ids = (const char *)(f.base + h.off_read_ids);
    f.blob = f.base + h.off_blob;
    madvise((void *)f.base, f.size, MADV_SEQUENTIAL);
    return ADB_OK;
}

// libzstd is present in the image without headers: bound at run time, only when a container asks for it
struct Zstd {
    void *lib = nullptr;
    size_t (*decompress)(void *, size_t, const void *, size_t) = nullptr;
    unsigned long long (*content_size)(const void *, size_t) = nullptr;
    unsigned (*is_error)(size_t) = nullptr;
    bool load() {
        if (decompress) return true;
        lib = dlopen("libzstd.so.1", RTLD_NOW | RTLD_LOCAL);
        if (!lib) return false;
        decompress = (decltype(decompress))dlsym(lib, "ZSTD_decompress");
        content_size = (decltype(content_size))dlsym(lib, "ZSTD_getFrameContentSize");
        is_error = (decltype(is_error))dlsym(lib, "ZSTD_isError");
        return decompress && content_size && is_error;
    }
};

template <class T>
struct Queue {
    std::mutex m;
    std::condition_variable cv;
    std::deque<T> q;
    void push(T v) { { std::lock_guard<std::mutex> l(m); q.push_back(v); } cv.notify_one(); }
    T pop() {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { return !q.empty(); });
        T v = q.front();
        q.pop_front();
        return v;
    }
};

struct Slot {
    // pinned host memory
    uint8_t *comp = nullptr;
    size_t comp_cap = 0;
    int64_t *coffs = nullptr, *foffs = nullptr;  // foffs: zstd frames of a device-decoded chunk
    int32_t *zfail = nullptr;                     // frames of the chunk the device refused
    int32_t *nsamp = nullptr, *lens = nullptr, *src_file = nullptr, *src_read = nullptr, *status = nullptr;
    float *coff = nullptr, *cscale = nullptr;
    char *ids = nullptr;
    adb_record *recs = nullptr;
    int nr = 0, nb = 0;
    size_t comp_bytes = 0, dec_bytes = 0;
    int svb = 1;  // 0: raw int16, 1: svb16 streams, 2: zstd frames of svb16 streams (decoded on the device)
    bool last = false;
    int error = 0;
    cudaEvent_t done = nullptr;
};

struct CopyJob { const uint8_t *src; uint8_t *dst; size_t bytes; size_t dst_cap; bool zstd; };

struct Table {  // one output file
    std::vector<adb_record> recs;
    std::vector<char> ids;  // [n][ID_SLOT_WIDTH + 1]
    std::map<int, std::vector<int32_t>> overflow;
    int index = 0;
    bool pass = true;
};

struct FileRing {
    std::vector<Slot> slots;
    int chunk_reads = 0, chunk_batches = 0;
    size_t comp_cap = 0;
};

static void file_ring_free(void *p) {
    FileRing *ring = (FileRing *)p;
    if (!ring) return;
    for (auto &s : ring->slots) {
        void *ps[] = {s.comp, s.coffs, s.foffs, s.zfail, s.nsamp, s.lens, s.src_file, s.src_read, s.status, s.coff, s.cscale, s.ids, s.recs};
        for (void *q : ps) if (q) cudaFreeHost(q);
        if (s.done) cudaEventDestroy(s.done);
    }
    delete ring;
}

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

}  // namespace adbf

extern "C" int adb_detect_files(adb_ctx *ctx, const adb_file_job *job, const adb_config *cfg, const float *cnn_weights,
                                adb_file_stats *stats) {
    using namespace adbf;
    if (!ctx || !job || !job->paths || job->n_paths < 0 || !stats || job->minibatch_size < 1 || job->batch_size_output < 1) {
        set_err("invalid argument");
        return ADB_ERR_ARG;
    }
    int rc = check_config(cfg);
    if (rc) return rc;
    if (cfg->primary_method == ADB_METHOD_CNN && !cnn_weights) { set_err("cnn_weights required"); return ADB_ERR_ARG; }
    memset(stats, 0, sizeof(*stats));
    const double t_start = now_s();
    const int m = cfg->sig_preload_size, mbs = job->minibatch_size;
    const int chunk_batches = std::max(1, job->chunk_batches > 0 ? job->chunk_batches : 16);
    const int chunk_reads = chunk_batches * mbs;
    // (measured on the 16-core box, 400 000 RNA004 reads: 4 / 8 / 12 copy threads -> 1.15 / 1.46 / 1.47 M reads/s file -> tables)
    int n_copy_thr = std::max(1, job->n_copy_threads > 0 ? job->n_copy_threads : (int)std::min(8u, std::max(2u, usable_cpus() / 2)));
    if (const char *e = getenv("ADB_COPY_THREADS")) n_copy_thr = std::max(1, atoi(e));  // (experiments)
    const int n_fmt_thr = std::max(1, job->n_format_threads > 0 ? job->n_format_threads : (int)std::min(16u, std::max(2u, std::thread::hardware_concurrency() / 2)));
    const bool write_csv = job->write_csv != 0 && job->out_dir != nullptr;

    std::vector<SigFile> files(job->n_paths);
    struct Closer { std::vector<SigFile> &f; ~Closer() { for (auto &x : f) x.close_(); } } closer{files};
    bool any_zstd = false;
    for (int i = 0; i < job->n_paths; i++) {
        rc = open_sigfile(job->paths[i], files[i]);
        if (rc) return rc;
        if (files[i].h.flags & F_ZSTD) any_zstd = true;
        for (uint64_t r = 0; r < files[i].h.n_reads; r++)
            if (files[i].nsamp[r] < 0) { set_err("negative n_samples in container"); return ADB_ERR_ARG; }
    }
    Zstd zstd;
    if (any_zstd && !zstd.load()) { set_err("container is zstd-compressed and libzstd.so.1 cannot be loaded"); return ADB_ERR_UNSUPPORTED; }

    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->twin) { rc = adb_ctx_create(ctx->device, &ctx->twin); if (rc) return rc; }
    ctx->twin->opt_no_fast_validate = ctx->opt_no_fast_validate;
        ctx->twin->opt_hist_validate = ctx->opt_hist_validate;
    ctx->twin->opt_cnn_fp32 = ctx->opt_cnn_fp32;
    ctx->twin->opt_exact_gsel = ctx->opt_exact_gsel;
        ctx->twin->opt_no_cand_followup = ctx->opt_no_cand_followup;
    adb_ctx *cc[2] = {ctx, ctx->twin};
    const float *w_devs[2] = {nullptr, nullptr};
    if (cfg->primary_method == ADB_METHOD_CNN)
        for (int k = 0; k < 2; k++) {
            if (cc[k]->h_misc2.ensure(sizeof(float) * ADB_CNN_NPARAMS)) { set_err("cudaMalloc weights"); return ADB_ERR_CUDA; }
            CUDA_TRY(cudaMemcpyAsync(cc[k]->h_misc2.p, cnn_weights, sizeof(float) * ADB_CNN_NPARAMS, cudaMemcpyHostToDevice, cc[k]->stream));
            w_devs[k] = (const float *)cc[k]->h_misc2.p;
        }

    // ---- the pinned ring (kept in the context between calls) ----
    const int n_slots = 4;
    const size_t per_read_cap = (size_t)m * 2 + (size_t)((m + 7) / 8 + 3) + 32;  // worst case of a stream / raw samples
    FileRing *ring = (FileRing *)ctx->file_ring;
    if (!ring || ring->chunk_reads < chunk_reads || ring->chunk_batches < chunk_batches || ring->comp_cap < per_read_cap * (size_t)chunk_reads + 64) {
        if (ring) { file_ring_free(ring); ctx->file_ring = nullptr; }
        ring = new FileRing();
        ring->slots.resize(n_slots);
        ring->chunk_reads = chunk_reads;
        ring->chunk_batches = chunk_batches;
        ring->comp_cap = per_read_cap * (size_t)chunk_reads + 64;
        ctx->file_ring = ring;
        ctx->file_ring_free = file_ring_free;
        for (auto &s : ring->slots) {
            s.comp_cap = ring->comp_cap;
            if (cudaHostAlloc((void **)&s.comp, s.comp_cap, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.coffs, sizeof(int64_t) * ((size_t)chunk_reads + 1), cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.foffs, sizeof(int64_t) * ((size_t)chunk_reads + 1), cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.zfail, sizeof(int32_t) * 4, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.nsamp, sizeof(int32_t) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.lens, sizeof(int32_t) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.src_file, sizeof(int32_t) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.src_read, sizeof(int32_t) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.status, sizeof(int32_t) * (size_t)chunk_batches, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.coff, sizeof(float) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.cscale, sizeof(float) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.ids, (size_t)(ID_SLOT_WIDTH + 1) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaHostAlloc((void **)&s.recs, sizeof(adb_record) * (size_t)chunk_reads, cudaHostAllocDefault) != cudaSuccess ||
                cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                file_ring_free(ring);
                ctx->file_ring = nullptr;
                set_err("cudaHostAlloc of the pinned ring failed");
                return ADB_ERR_CUDA;
            }
        }
    }
    std::vector<Slot> &slots = ring->slots;
    Queue<Slot *> q_free, q_filled, q_inflight;
    for (auto &s : slots) q_free.push(&s);
    std::atomic<int> failed{0};
    std::string fail_msg;
    std::mutex fail_m;
    auto fail = [&](int code, const std::string &msg) {
        std::lock_guard<std::mutex> l(fail_m);
        if (!failed.load()) { fail_msg = msg; failed.store(code); }
    };
    double read_s = 0.0, write_s = 0.0, gpu_wait_s = 0.0;
    std::atomic<long long> comp_total{0}, host_frames{0};
    const bool device_zstd = !ctx->opt_host_zstd;

    // ---- reader ----
    std::thread reader([&]() {
        std::vector<CopyJob> jobs;
        Slot *s = q_free.pop();
        s->nr = 0; s->comp_bytes = 0; s->dec_bytes = 0; s->last = false; s->error = 0;
        s->svb = 1;
        auto flush = [&](bool last) {
            const double t0 = now_s();
            s->nb = (s->nr + mbs - 1) / mbs;
            s->last = last;
            // the copies of the chunk, spread over the copy threads (large runs are cut)
            std::vector<CopyJob> cut;
            const size_t piece = 8u << 20;
            for (const CopyJob &j : jobs) {
                if (j.zstd || j.bytes <= piece) { cut.push_back(j); continue; }
                for (size_t o = 0; o < j.bytes; o += piece) cut.push_back({j.src + o, j.dst + o, std::min(piece, j.bytes - o), 0, false});
            }
            std::atomic<size_t> next{0};
            auto work = [&]() {
                for (;;) {
                    const size_t k = next.fetch_add(1);
                    if (k >= cut.size()) break;
                    const CopyJob &j = cut[k];
                    if (j.zstd) {
                        host_frames++;
                        const size_t got = zstd.decompress(j.dst, j.dst_cap, j.src, j.bytes);
                        if (zstd.is_error(got) || got != j.dst_cap) fail(ADB_ERR_ARG, "zstd frame of a read does not decompress to its stated size");
                    } else {
                        memcpy(j.dst, j.src, j.bytes);
                    }
                }
            };
            std::vector<std::thread> pool;
            const int nt = (int)std::min<size_t>(n_copy_thr, cut.size());
            for (int t = 1; t < nt; t++) pool.emplace_back(work);
            work();
            for (auto &t : pool) t.join();
            jobs.clear();
            if (s->svb == 1) memset(s->comp + s->comp_bytes, 0, 16);  // the slack behind the last stream
            comp_total += (long long)s->comp_bytes;
            read_s += now_s() - t0;
            q_filled.push(s);
            if (!last) {
                s = q_free.pop();
                s->nr = 0; s->comp_bytes = 0; s->dec_bytes = 0; s->last = false; s->error = 0; s->svb = 1;
            }
        };
        for (int fi = 0; fi < (int)files.size() && !failed.load(); fi++) {
            const SigFile &f = files[fi];
            const uint8_t *keep = job->keep ? job->keep[fi] : nullptr;
            const bool svb = (f.h.flags & F_SVB16) != 0, zs = (f.h.flags & F_ZSTD) != 0;
            const int idw = (int)f.h.id_width;
            for (int64_t r = 0; r < (int64_t)f.h.n_reads && !failed.load(); r++) {
                if (keep && !keep[r]) continue;
                const int64_t o0 = f.coffs[r], o1 = f.coffs[r + 1];
                if (o0 < 0 || o1 < o0 || (uint64_t)o1 > f.h.blob_bytes) { fail(ADB_ERR_ARG, "stream offsets outside the container blob"); break; }
                int ns = std::min(f.nsamp[r], m);
                size_t bytes = (size_t)(o1 - o0), dst_bytes = bytes;
                const uint8_t *src = f.blob + o0;
                // an svb16 stream in one zstd frame that the device takes travels as it is (no host decompression)
                uint64_t zcs = 0;
                const bool zdev = zs && svb && device_zstd && zstd_screen(src, bytes, per_read_cap * 4, &zcs);
                const int rep = zdev ? 2 : (svb ? 1 : 0);
                if (s->nr > 0 && s->svb != rep) flush(false);  // a chunk holds one representation
                s->svb = rep;
                const int k = s->nr;
                if (zdev) {
                    if (f.nsamp[r] > m) { fail(ADB_ERR_UNSUPPORTED, "compressed read longer than sig_preload_size in the container"); break; }
                    const size_t dst_off = s->comp_bytes, dec_off = s->dec_bytes;
                    if (dst_off + bytes + 32 > s->comp_cap) { fail(ADB_ERR_ARG, "a read's stream exceeds the worst-case size for its sample count"); break; }
                    const bool extend = !jobs.empty() && !jobs.back().zstd && jobs.back().src + jobs.back().bytes == src &&
                                        jobs.back().dst + jobs.back().bytes == s->comp + dst_off;
                    if (extend) jobs.back().bytes += bytes;
                    else jobs.push_back({src, s->comp + dst_off, bytes, bytes, false});
                    s->foffs[k] = (int64_t)dst_off;
                    s->comp_bytes = dst_off + bytes;
                    s->foffs[k + 1] = (int64_t)s->comp_bytes;
                    s->coffs[k] = (int64_t)dec_off;
                    s->dec_bytes = dec_off + (size_t)((zcs + 15) & ~(uint64_t)15);
                    s->coffs[k + 1] = (int64_t)s->dec_bytes;
                } else {
                if (zs) {
                    const unsigned long long cs = zstd.content_size(src, bytes);
                    if (cs == (unsigned long long)-1 || cs == (unsigned long long)-2 || cs > per_read_cap * 4) { fail(ADB_ERR_ARG, "zstd frame without a usable content size"); break; }
                    dst_bytes = (size_t)cs;
                }
                if (!svb) {  // raw int16 samples: only the preload window travels
                    dst_bytes = std::min(dst_bytes, (size_t)ns * 2);
                    if (!zs) bytes = dst_bytes;
                    ns = (int)(dst_bytes / 2);
                } else if (f.nsamp[r] > m) {
                    // a stream longer than the preload window cannot be cut without decoding: containers are written with
                    // the window applied (adapted_b200.ingest.write_container_v2 truncates)
                    fail(ADB_ERR_UNSUPPORTED, "compressed read longer than sig_preload_size in the container");
                    break;
                }
                const size_t dst_off = svb ? ((s->comp_bytes + 15) & ~(size_t)15) : s->comp_bytes;
                if (dst_off + dst_bytes + 32 > s->comp_cap) { fail(ADB_ERR_ARG, "a read's stream exceeds the worst-case size for its sample count"); break; }
                // consecutive uncompressed streams of one file form one run (16-byte aligned in the file as in the slot)
                const bool extend = !zs && !jobs.empty() && !jobs.back().zstd && jobs.back().src + jobs.back().bytes == src &&
                                    jobs.back().dst + jobs.back().bytes == s->comp + dst_off;
                if (extend) jobs.back().bytes += bytes;
                else jobs.push_back({src, s->comp + dst_off, bytes, dst_bytes, zs});
                s->coffs[k] = svb ? (int64_t)dst_off : (int64_t)(dst_off / 2);
                s->comp_bytes = dst_off + dst_bytes;
                s->coffs[k + 1] = svb ? (int64_t)((s->comp_bytes + 15) & ~(size_t)15) : (int64_t)(s->comp_bytes / 2);
                }
                s->nsamp[k] = ns;
                s->lens[k] = f.lens[r];
                s->coff[k] = f.coff[r];
                s->cscale[k] = f.cscale[r];
                s->src_file[k] = fi;
                s->src_read[k] = (int32_t)r;
                char *id = s->ids + (size_t)k * (ID_SLOT_WIDTH + 1);
                memcpy(id, f.ids + (size_t)r * idw, idw);
                id[idw] = 0;
                s->nr = k + 1;
                if (s->nr == chunk_reads) flush(false);
            }
        }
        if (failed.load()) s->error = 1;
        flush(true);
    });

    // ---- formatter pool + writer ----
    Queue<Table *> q_tables;
    std::atomic<long long> n_files{0};
    const std::string out_dir = job->out_dir ? job->out_dir : "";
    const char *llr_log = cfg->primary_method == ADB_METHOD_LLR ? "" : nullptr;
    std::vector<std::thread> formatters;
    if (write_csv) {
        const std::string d1 = out_dir + "/boundaries", d2 = out_dir + "/failed_reads";
        mkdir(out_dir.c_str(), 0777); mkdir(d1.c_str(), 0777); mkdir(d2.c_str(), 0777);
        for (int t = 0; t < n_fmt_thr; t++)
            formatters.emplace_back([&]() {
                std::vector<char> text;
                std::vector<const char *> idp;
                for (;;) {
                    Table *tb = q_tables.pop();
                    if (!tb) break;
                    const int n = (int)tb->recs.size();
                    idp.resize(n);
                    for (int i = 0; i < n; i++) idp[i] = tb->ids.data() + (size_t)i * (ID_SLOT_WIDTH + 1);
                    std::vector<int32_t> op_index, op_pos;
                    std::vector<int64_t> op_offs;
                    if (!tb->overflow.empty()) {
                        op_index.assign(n, -1);
                        op_offs.push_back(0);
                        int row = 0;
                        for (auto &kv : tb->overflow) {
                            op_index[kv.first] = row++;
                            op_pos.insert(op_pos.end(), kv.second.begin(), kv.second.end());
                            op_offs.push_back((int64_t)op_pos.size());
                        }
                        if (op_pos.empty()) op_pos.push_back(0);
                    }
                    text.resize((size_t)n * 448 + 4096);
                    int64_t len;
                    for (;;) {
                        len = adb_format_csv_ex(tb->recs.data(), nullptr, n, idp.data(), cfg->primary_method, llr_log, tb->pass ? 0 : 1,
                                                op_index.empty() ? nullptr : op_index.data(), op_offs.empty() ? nullptr : op_offs.data(),
                                                op_pos.empty() ? nullptr : op_pos.data(), text.data(), (int64_t)text.size());
                        if (len < 0 || len <= (int64_t)text.size()) break;
                        text.resize((size_t)len);
                    }
                    if (len < 0) fail((int)len, "adb_format_csv_ex failed");
                    else {
                        const std::string fn = out_dir + (tb->pass ? "/boundaries/detected_boundaries_" : "/failed_reads/failed_reads_") +
                                               std::to_string(tb->index) + ".csv";
                        FILE *fp = fopen(fn.c_str(), "wb");
                        if (!fp || fwrite(text.data(), 1, (size_t)len, fp) != (size_t)len) fail(ADB_ERR_ARG, "cannot write " + fn);
                        if (fp) fclose(fp);
                        n_files++;
                    }
                    delete tb;
                }
            });
    }
    adb_ctx *aux_ctx = nullptr;  // the rare overflow reads (open-pore lists beyond the record) are redone here
    std::thread writer([&]() {
        Table *acc[2] = {new Table(), new Table()};  // [0] fail, [1] pass
        int bidx[2] = {job->bidx_fail, job->bidx_pass};
        auto emit = [&](int key, size_t n) {
            Table *t = acc[key];
            Table *out = new Table();
            out->pass = key == 1;
            out->index = bidx[key]++;
            out->recs.assign(t->recs.begin(), t->recs.begin() + n);
            out->ids.assign(t->ids.begin(), t->ids.begin() + n * (ID_SLOT_WIDTH + 1));
            Table *rest = new Table();
            rest->recs.assign(t->recs.begin() + n, t->recs.end());
            rest->ids.assign(t->ids.begin() + n * (ID_SLOT_WIDTH + 1), t->ids.end());
            for (auto &kv : t->overflow) {
                if ((size_t)kv.first < n) out->overflow[kv.first] = std::move(kv.second);
                else rest->overflow[kv.first - (int)n] = std::move(kv.second);
            }
            delete t;
            acc[key] = rest;
            if (write_csv) q_tables.push(out); else delete out;
        };
        for (;;) {
            Slot *s = q_inflight.pop();
            const double t0 = now_s();
            if (s->nr > 0 && !s->error && cudaEventSynchronize(s->done) != cudaSuccess) fail(ADB_ERR_CUDA, "cudaEventSynchronize failed in the writer");
            gpu_wait_s += now_s() - t0;
            const double t1 = now_s();
            if (!s->error && s->nr > 0 && s->svb == 2 && *s->zfail != 0)
                fail(ADB_ERR_ARG, "zstd frame of a read does not decompress to its stated size");
            if (!s->error && !failed.load()) {
                for (int b = 0; b < s->nb; b++) {
                    const int a = b * mbs, e = std::min(s->nr, a + mbs);
                    if (s->status[b] != ADB_OK) {  // the reference loses the minibatch (handle_completed_future, file_proc.py:726-731)
                        stats->lost += e - a;
                        continue;
                    }
                    for (int i = a; i < e; i++) {
                        const adb_record &r = s->recs[i];
                        const int key = r.success ? 1 : 0;
                        Table *t = acc[key];
                        if ((r.valid & ADB_V_FIELDS) && (r.valid & ADB_V_OPEN_PORES) && r.n_open_pores > ADB_MAX_OPEN_PORES && write_csv) {
                            // full list from the GPU: decode the read's stream again and scan it (adb_open_pores_host)
                            const SigFile &f = files[s->src_file[i]];
                            const int64_t rr = s->src_read[i];
                            std::vector<int32_t> list;
                            int orc = ADB_OK;
                            if (!aux_ctx) orc = adb_ctx_create(ctx->device, &aux_ctx);
                            std::vector<int16_t> samples((size_t)std::max(s->nsamp[i], 1));
                            std::vector<uint8_t> stream;
                            if (!orc) {
                                const uint8_t *src = f.blob + f.coffs[rr];
                                size_t bytes = (size_t)(f.coffs[rr + 1] - f.coffs[rr]);
                                if (f.h.flags & F_ZSTD) {
                                    stream.resize((size_t)zstd.content_size(src, bytes) + 32);
                                    bytes = zstd.decompress(stream.data(), stream.size(), src, bytes);
                                } else {
                                    stream.assign(src, src + bytes);
                                    stream.resize(bytes + 32);
                                }
                                if (f.h.flags & F_SVB16) {
                                    // 16-byte aligned copy with slack, as the decoder expects
                                    std::vector<uint8_t> al(stream.size() + 48);
                                    uint8_t *p = (uint8_t *)(((uintptr_t)al.data() + 15) & ~(uintptr_t)15);
                                    memcpy(p, stream.data(), bytes);
                                    const int64_t co[2] = {0, (int64_t)((bytes + 15) & ~(size_t)15)};
                                    const float zero = 0.f;
                                    adb_svb_batch sb;
                                    memset(&sb, 0, sizeof sb);
                                    sb.comp = p; sb.comp_offsets = co; sb.n_samples = &s->nsamp[i]; sb.n_reads = 1; sb.m = m; sb.batch_size = 1;
                                    sb.full_lens = &s->lens[i]; sb.calib_offset = &zero; sb.calib_scale = &zero;
                                    orc = adb_svb16_decode_host(aux_ctx, &sb, samples.data());
                                } else {
                                    memcpy(samples.data(), stream.data(), (size_t)s->nsamp[i] * 2);
                                }
                            }
                            if (!orc) {
                                const int64_t off2[2] = {0, s->nsamp[i]};
                                adb_batch ob;
                                ob.signal = samples.data(); ob.sig_type = ADB_SIG_I16; ob.n_reads = 1; ob.m = m; ob.batch_size = 1;
                                ob.offsets = off2; ob.full_lens = &s->lens[i]; ob.calib_offset = &s->coff[i]; ob.calib_scale = &s->cscale[i];
                                const int32_t sel0 = 0, sb0 = 0, se0 = r.primary_adapter_end;
                                int64_t oo[2] = {0, 0};
                                orc = adb_open_pores_host(aux_ctx, &ob, &sel0, 1, &sb0, &se0, oo, nullptr, 0);
                                if (!orc) {
                                    list.resize((size_t)std::max<int64_t>(oo[1], 1));
                                    orc = adb_open_pores_host(aux_ctx, &ob, &sel0, 1, &sb0, &se0, oo, list.data(), (int64_t)list.size());
                                    list.resize((size_t)oo[1]);
                                }
                            }
                            if (orc) fail(orc, "open-pore overflow pass failed: " + adb_err_string());
                            t->overflow[(int)t->recs.size()] = std::move(list);
                        }
                        t->recs.push_back(r);
                        const char *id = s->ids + (size_t)i * (ID_SLOT_WIDTH + 1);
                        t->ids.insert(t->ids.end(), id, id + ID_SLOT_WIDTH + 1);
                        if (r.success) stats->pass++; else stats->fail++;
                        if ((int)t->recs.size() >= job->batch_size_output) emit(key, (size_t)job->batch_size_output);
                    }
                }
                stats->reads += s->nr;
            }
            write_s += now_s() - t1;
            const bool last = s->last;
            q_free.push(s);
            if (last) break;
        }
        // the remainders, fail table first like the reference's savers finish (order is immaterial: separate files)
        for (int key = 0; key < 2; key++) {
            if (!acc[key]->recs.empty() && !failed.load()) emit(key, acc[key]->recs.size());
            delete acc[key];
        }
    });

    // ---- GPU thread (this one) ----
    cudaStream_t cs = ctx->copy_stream;
    int ch = 0;
    long long h2d_bytes = 0;
    for (;; ch++) {
        Slot *s = q_filled.pop();
        adb_ctx *c = cc[ch & 1];
        cudaStream_t ks = c->stream;
        const int nr = s->nr;
        if (nr > 0 && !s->error && !failed.load()) {
            int e = ADB_OK;
            auto step = [&]() -> int {
                // the device buffers of this context are free once its previous chunk has finished
                if (ch >= 2) CUDA_TRY(cudaEventSynchronize(c->p_done[0]));
                const size_t cbytes = s->comp_bytes + 16;
                size_t dec_samples = 0;
                // (the svb16 streams of a zstd chunk are laid out in p_comp after the zstd decode)
                for (int i = 0; i < nr; i++) dec_samples += (size_t)s->nsamp[i];
                if (c->p_comp[0].ensure(cbytes + 64) || c->p_coffs[0].ensure(sizeof(int64_t) * ((size_t)nr + 1)) ||
                    c->p_nsamp[0].ensure(sizeof(int32_t) * (size_t)nr + 16) || c->p_signal[0].ensure(dec_samples * 2 + 64) ||
                    c->p_offsets[0].ensure(sizeof(int64_t) * ((size_t)nr + 1)) || c->p_lens[0].ensure(sizeof(int32_t) * (size_t)nr + 16) ||
                    c->p_coff[0].ensure(sizeof(float) * (size_t)nr + 16) || c->p_cscale[0].ensure(sizeof(float) * (size_t)nr + 16) ||
                    c->p_records[0].ensure(sizeof(adb_record) * (size_t)nr) || c->p_status[0].ensure(sizeof(int) * (size_t)s->nb + 16)) {
                    set_err("cudaMalloc pipeline staging");
                    return ADB_ERR_CUDA;
                }
                if (s->svb == 2) {  // zstd frames -> zstd_decode_kernel -> svb16 streams in p_comp
                    if (c->p_frames[0].ensure(s->comp_bytes + 16) || c->p_foffs[0].ensure(sizeof(int64_t) * ((size_t)nr + 1)) ||
                        c->p_comp[0].ensure(s->dec_bytes + 64) || c->p_zstat[0].ensure(sizeof(int32_t) * (size_t)nr + 16) ||
                        c->z_fail.ensure(16)) {
                        set_err("cudaMalloc pipeline staging");
                        return ADB_ERR_CUDA;
                    }
                    CUDA_TRY(cudaMemcpyAsync(c->p_frames[0].p, s->comp, s->comp_bytes, cudaMemcpyHostToDevice, cs));
                    CUDA_TRY(cudaMemcpyAsync(c->p_foffs[0].p, s->foffs, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
                    CUDA_TRY(cudaMemcpyAsync(c->p_coffs[0].p, s->coffs, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
                    h2d_bytes += (long long)(s->comp_bytes + (size_t)nr * 8);
                } else {
                    void *sig_dst = s->svb ? c->p_comp[0].p : c->p_signal[0].p;
                    CUDA_TRY(cudaMemcpyAsync(sig_dst, s->comp, s->svb ? cbytes : s->comp_bytes, cudaMemcpyHostToDevice, cs));
                    CUDA_TRY(cudaMemcpyAsync(s->svb ? c->p_coffs[0].p : c->p_offsets[0].p, s->coffs, sizeof(int64_t) * ((size_t)nr + 1), cudaMemcpyHostToDevice, cs));
                    h2d_bytes += (long long)cbytes;
                }
                CUDA_TRY(cudaMemcpyAsync(c->p_nsamp[0].p, s->nsamp, sizeof(int32_t) * (size_t)nr, cudaMemcpyHostToDevice, cs));
                CUDA_TRY(cudaMemcpyAsync(c->p_lens[0].p, s->lens, sizeof(int32_t) * (size_t)nr, cudaMemcpyHostToDevice, cs));
                CUDA_TRY(cudaMemcpyAsync(c->p_coff[0].p, s->coff, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
                CUDA_TRY(cudaMemcpyAsync(c->p_cscale[0].p, s->cscale, sizeof(float) * (size_t)nr, cudaMemcpyHostToDevice, cs));
                CUDA_TRY(cudaEventRecord(c->p_copied[0], cs));
                CUDA_TRY(cudaStreamWaitEvent(ks, c->p_copied[0], 0));
                h2d_bytes += (long long)((size_t)nr * 28);
                if (s->svb == 2) {
                    CUDA_TRY(cudaMemsetAsync(c->z_fail.p, 0, sizeof(int32_t), ks));
                    CUDA_TRY(cudaMemsetAsync((uint8_t *)c->p_comp[0].p + s->dec_bytes, 0, 16, ks));  // the slack behind the last stream
                    int r1 = launch_zstd_decode(c, (const uint8_t *)c->p_frames[0].p, (const int64_t *)c->p_foffs[0].p, (uint8_t *)c->p_comp[0].p,
                                                (const int64_t *)c->p_coffs[0].p, (int32_t *)c->p_zstat[0].p, (int32_t *)c->z_fail.p, nr, ks);
                    if (r1) return r1;
                    CUDA_TRY(cudaMemcpyAsync(s->zfail, c->z_fail.p, sizeof(int32_t), cudaMemcpyDeviceToHost, ks));
                }
                if (s->svb) {
                    int r2 = launch_svb_decode(c, (const uint8_t *)c->p_comp[0].p, (const int64_t *)c->p_coffs[0].p,
                                               (const int32_t *)c->p_nsamp[0].p, nr, (int64_t *)c->p_offsets[0].p,
                                               (int16_t *)c->p_signal[0].p, ks);
                    if (r2) return r2;
                }
                adb_batch d;
                d.signal = c->p_signal[0].p; d.sig_type = ADB_SIG_I16; d.n_reads = nr; d.m = m; d.batch_size = mbs;
                d.offsets = (const int64_t *)c->p_offsets[0].p; d.full_lens = (const int32_t *)c->p_lens[0].p;
                d.calib_offset = (const float *)c->p_coff[0].p; d.calib_scale = (const float *)c->p_cscale[0].p;
                int r3 = adb_detect_dev(c, &d, cfg, w_devs[ch & 1], (adb_record *)c->p_records[0].p, (int *)c->p_status[0].p, ks);
                if (r3) return r3;
                CUDA_TRY(cudaMemcpyAsync(s->recs, c->p_records[0].p, sizeof(adb_record) * (size_t)nr, cudaMemcpyDeviceToHost, ks));
                CUDA_TRY(cudaMemcpyAsync(s->status, c->p_status[0].p, sizeof(int) * (size_t)s->nb, cudaMemcpyDeviceToHost, ks));
                CUDA_TRY(cudaEventRecord(c->p_done[0], ks));
                CUDA_TRY(cudaEventRecord(s->done, ks));
                return ADB_OK;
            };
            e = step();
            if (e) { fail(e, adb_err_string()); s->error = 1; }
        } else if (failed.load()) {
            s->error = 1;
        }
        const bool last = s->last;
        q_inflight.push(s);
        if (last) break;
    }
    reader.join();
    writer.join();
    for (size_t t = 0; t < formatters.size(); t++) q_tables.push(nullptr);
    for (auto &t : formatters) t.join();
    cudaStreamSynchronize(cs);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->twin->stream);
    if (aux_ctx) adb_ctx_destroy(aux_ctx);
    stats->files = n_files.load();
    stats->comp_bytes = comp_total.load();
    stats->h2d_bytes = h2d_bytes;
    ctx->zstd_host_frames = host_frames.load();
    stats->seconds = now_s() - t_start;
    stats->read_s = read_s;
    stats->gpu_wait_s = gpu_wait_s;
    stats->write_s = write_s;
    if (failed.load()) {
        set_err(fail_msg);
        return failed.load();
    }
    return ADB_OK;
}
