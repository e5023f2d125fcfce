// capi.cu — the extern "C" layer of libgbin.so: context, HBM workspace and the pipeline
//   scan (process_read, binning.c:918-1040) -> sort (zhash grouping, :1044-1069) -> run-length + prune (:1085-1144).
// There is no CPU fallback anywhere in this file: every entry point either runs the CUDA kernels or
// returns an error code.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gbin.h"
#include "gbin_internal.h"
#include "prefix_scan.cuh"

using namespace gbin;

namespace {

struct DevBuf {  // frees its memory when destroyed (with the context that holds it)
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 16 + 256;  // a little slack so near-equal batches do not reallocate
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    // grows like ensure() but keeps the first `keep` bytes (the parts of a table that earlier passes of a batch have written)
    cudaError_t ensure_keep(size_t bytes, size_t keep, cudaStream_t st) {
        if (bytes <= cap) return cudaSuccess;
        if (!p || keep == 0) return ensure(bytes);
        void *q = nullptr;
        const size_t want = bytes + bytes / 16 + 256;
        cudaError_t e = cudaMalloc(&q, want);
        if (e != cudaSuccess) return e;
        e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        cudaFree(p);
        p = q;
        cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};

struct HostBuf {  // page-locked; freed when destroyed
    void *p = nullptr;
    size_t cap = 0;
    HostBuf() = default;
    HostBuf(const HostBuf &) = delete;
    HostBuf &operator=(const HostBuf &) = delete;
    ~HostBuf() { release(); }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Small device-resident scalars (ctx->misc) and their pinned host mirror (ctx->h_misc).  Values the host needs at the same
// point are grouped into one member, so that read_back() fetches them in one copy.
struct Misc {
    struct {
        GroupCounts counts;
        unsigned long long bad_bases;  // of pipeline 1's scan
    } grp;
    struct {
        unsigned long long total_windows;
        unsigned int max_len;
    } reads;
    uint64_t part_counts[256];
    // super-k-mer pipelines (2 and 3)
    unsigned long long skr_counters[4];  // [0] bad bases, [1] records, [2] instances
    uint32_t skr_ticket, n_buckets_dev;
    struct {
        uint32_t n_inst, n_runs;
    } plan;
    unsigned long long chunk_totals[SKR_MAX_CHUNKS];
    // pipeline 2
    SkrGroupCounters gc;
    uint32_t chunk_tickets[SKR_MAX_CHUNKS];
    // pipeline 3
    V3Counters gc3;
    unsigned long long n_mmers;         // distinct m-mer codes of a batch (automatic key layout)
    unsigned long long n_real_entries;  // entries of the sort that are not empty pieces
    uint32_t chunk_bounds[SKR_MAX_CHUNKS + 1];
    uint32_t v3_tickets[2 * SKR_MAX_CHUNKS];
    unsigned long long lsd_totals[SKR_MAX_CHUNKS];
    uint64_t v3_chunk_sum;
    // file path and table digest
    uint32_t split_n_nl, split_n_reads;
    char last_byte;                     // of the file image
    unsigned long long digest;
};

// Host path only.  HostFeed: the reads are still in host memory; the scan stage copies them chunk by chunk on the copy
// stream and scans every chunk as soon as it has landed.  HostSink: pinned destinations for the big arrays of the
// table; finished chunks of the grouping are copied out on the second copy stream while later chunks are still running.
struct HostFeed {
    const char *src;     // host
    char *dst;           // device
    uint64_t bytes;
    int chunks;
};
struct HostSink {
    uint64_t *kmer_codes, *kmer_id_off;  // pinned; capacities in k-mers
    int32_t *read_ids;                   // pinned; capacity in ids
    uint64_t kmer_cap, id_cap;
    uint64_t kmers_done, ids_done;       // what has been enqueued for copy so far
    int chunks;
};

// Timing events of one call, in the order they are recorded.
enum : int { EV_START, EV_READS_ON_DEVICE, EV_SCANNED, EV_SORTED, EV_GROUPED, EV_TABLE_ON_HOST, EV_COUNT };

}  // namespace

struct gbin_ctx {
    gbin_config cfg;
    int KW;
    int sm_count;
    cudaStream_t stream;
    cudaStream_t st_h2d, st_d2h;  // copy streams of the host path (H2D of later read chunks / D2H of finished table chunks overlap the kernels)
    cudaEvent_t ev_feed[SKR_MAX_CHUNKS], ev_chunk[SKR_MAX_CHUNKS], ev_copy;
    cudaStream_t st_aux;          // second compute stream of pipeline 3's grouping stage
    cudaEvent_t ev_fork, ev_join;
    int host_chunks;              // GBIN_HOST_CHUNKS (default 8; 1 = no overlap)
    char err[512];
    gbin_timings tm;
    cudaEvent_t ev[EV_COUNT];
    // inputs staged by the host path
    DevBuf d_reads, d_starts, d_lens, d_ids;
    // pipeline workspace
    DevBuf rec_a, rec_b, radix_scratch, win_counts, rec_off, scan_scratch;
    DevBuf group_of, run_start, surv_index, id_offset, surv_group, bucket_of;
    DevBuf misc;
    // workspace of the super-k-mer pipelines (2 and 3)
    DevBuf skr_a, skr_b, tile_state, inst_prefix, run_excl, skr_run_start, small_prefix, unit_base, units, unit_state, o_kmer_mmer, bucket_excl, big_list, big_k0, big_k1, big_arr, stg_ids, stg_codes, stg_mmer, stg_off, skr_side;
    // pipeline 3 workspace
    DevBuf ent_a, ent_b, piece_n, sorted_info, v3_base64, v3_head_run, v3_unit_out, v3_unit_excl, v3_atoms, v3_lsd_aux, v3_bitmap;
    DevBuf x_list_off, x_ids;         // gbin_expand_read_ids_device's result
    void *donated = nullptr;          // gbin_donate_scratch: caller-owned device memory the next grouping call may use for its sort buffers
    uint64_t donated_bytes = 0;
    bool v3_lsd_seen = false;         // a batch on this context had long spans: keep the arrays of their global sort
    uint64_t v3_lsd_cap_seen = 0;     // and how many k-mers they were sized for
    uint64_t v3_pass_max = 2000000000ull;  // k-mer instances per pass of pipeline 3 (gbin_set_tuning "v3_pass_max")
    uint64_t v3_auto_n = 0;           // record count for which the key layout below was chosen (v3_nc == 0: automatic)
    int v3_auto_h = 0, v3_auto_nc = 1;
    int v3_h, v3_nc, v3_cap;  // key layout and unit capacity of pipeline 3 (gbin_set_tuning; GBIN_V3_H / GBIN_V3_NC / GBIN_V3_CAP); v3_cap 0 = by layout
    int v3_cap_eff;           // the capacity of the current batch
    int xchg_timeout_ms = 120000;  // gbin_set_tuning "xchg_timeout_ms" / GBIN_XCHG_TIMEOUT_MS
    int pipeline;        // 3: sort by reference + warp units, falling back to 2, then 1 (default); 2: super-k-mer path with v1 as fallback; 1: v1 only
    int last_pipeline;   // which one produced the last table
    uint32_t fallbacks;  // fallbacks to the next pipeline (3 -> 2 -> 1) since creation
    gbin_run_stats rs;   // sizes seen by the last pipeline-2 or pipeline-3 run
    // owner exchange over peer memory (multi-GPU, one process per GPU)
    struct {
        bool created = false, attached = false;
        uint32_t rank = 0, world = 0, epoch = 0;
        uint64_t cap = 0;
        void *recv = nullptr;
        XchgShared *sh = nullptr;
        char **dst_tab = nullptr;
        XchgResult *result = nullptr;
        XchgPlan plan;
        void *opened[2 * XCHG_MAX_WORLD];
        int n_opened = 0;
    } xg;
    // device-resident result
    DevBuf o_mmer_codes, o_mmer_kmer_off, o_kmer_codes, o_kmer_id_off, o_read_ids;
    // pinned host arena for results of the host path + small readbacks
    HostBuf h_misc, h_result, h_kmer_codes, h_kmer_id_off, h_read_ids, h_file;
    DevBuf split_nl, split_tiles_buf, split_base;  // device-side fgets splitting
    KernelProf prof;
};

namespace {

int fail(gbin_ctx *ctx, int code, const char *fmt, ...) {
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) {                                                                             \
            (void)cudaGetLastError();                                                                         \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? GBIN_E_NOMEM : GBIN_E_CUDA, "%s: %s (%s:%d)", \
                        #call, cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
        }                                                                                                     \
    } while (0)

int check_config(const gbin_config *c) {
    if (!c) return GBIN_E_INVALID_ARG;
    const int K = c->kmer_size, M = c->mmer_size;
    if (M < 2 || M > 15) return GBIN_E_INVALID_CONFIG;       // int scores (binning.c:911) hold 4^15-1 at most
    if (K < 2 * M || K > 64) return GBIN_E_INVALID_CONFIG;   // binning.c:997 is dead code only for K >= 2M
    return GBIN_OK;
}

// Makes the context's device current and picks the call's stream: the caller's, else the context's own.
cudaError_t begin_call(gbin_ctx *ctx, void *stream, cudaStream_t *st) {
    *st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return cudaSetDevice(ctx->cfg.device);
}

// Copies one member of the device scalars into the pinned mirror and waits for it: one host round trip.
template <typename T>
cudaError_t read_back(gbin_ctx *ctx, T Misc::*field, cudaStream_t st) {
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    const cudaError_t e = cudaMemcpyAsync(&(hm->*field), &(dm->*field), sizeof(T), cudaMemcpyDeviceToHost, st);
    return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
}

// The device table over the context's output arrays.
gbin_table device_table(const gbin_ctx *ctx, uint64_t n_instances, uint64_t n_distinct, uint64_t S, uint64_t NS, uint64_t B) {
    gbin_table t;
    memset(&t, 0, sizeof t);
    t.kmer_size = ctx->cfg.kmer_size;
    t.mmer_size = ctx->cfg.mmer_size;
    t.abundance_cutoff = ctx->cfg.abundance_cutoff;
    t.kmer_words = ctx->KW;
    t.on_device = 1;
    t.ctx_owned = 1;
    t.n_instances = n_instances;
    t.n_distinct = n_distinct;
    t.n_kmers = S;
    t.n_ids = NS;
    t.n_buckets = B;
    t.mmer_codes = ctx->o_mmer_codes.as<uint32_t>();
    t.mmer_kmer_off = ctx->o_mmer_kmer_off.as<uint64_t>();
    t.kmer_codes = ctx->o_kmer_codes.as<uint64_t>();
    t.kmer_id_off = ctx->o_kmer_id_off.as<uint64_t>();
    t.read_ids = ctx->o_read_ids.as<int32_t>();
    return t;
}

// Bucket directory of the super-k-mer pipelines over the S surviving k-mers in ctx->o_kmer_mmer; *B receives the bucket count.
int emit_bucket_directory(gbin_ctx *ctx, uint64_t S, uint64_t NS, cudaStream_t st, int *launches, uint64_t *B) {
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    CU(ctx->bucket_excl.ensure((S + 1) * 4));
    CU(ctx->o_mmer_codes.ensure((S + 1) * sizeof(uint32_t)));
    CU(ctx->o_mmer_kmer_off.ensure((S + 2) * sizeof(uint64_t)));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(S + 1024)));
    const bool on = ctx->prof.begin(KK_EMIT, st);
    const int lp = skr_emit_buckets(ctx->o_kmer_mmer.as<uint32_t>(), S, NS, ctx->bucket_excl.as<uint32_t>(), ctx->scan_scratch.as<uint32_t>(),
                                    ctx->o_mmer_codes.as<uint32_t>(), ctx->o_mmer_kmer_off.as<uint64_t>(), ctx->o_kmer_id_off.as<uint64_t>(),
                                    &dm->n_buckets_dev, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::n_buckets_dev, st));
    *B = hm->n_buckets_dev;
    return GBIN_OK;
}

// Host path: streams the finished part of the table to the host while later chunks are grouped.  The table is written in
// unit order, and what the units of chunk c wrote is final once ctx->ev_chunk[c] has fired; totals_host[c] then holds
// {k-mers << shift | ids} written up to the end of chunk c.  A chunk with k-mers left to pipeline 3's global sort for long spans
// (lsd_totals_host[c] != 0) ends the streaming, as does an arena too small: the rest is copied at the end.
int stream_finished_chunks(gbin_ctx *ctx, HostSink *sink, uint32_t n, const unsigned long long *totals_host, int shift,
                           const unsigned long long *lsd_totals_host) {
    const int KW = ctx->KW;
    for (uint32_t c = 0; c < n; c++) {
        CU(cudaEventSynchronize(ctx->ev_chunk[c]));
        if (lsd_totals_host && lsd_totals_host[c]) break;
        const unsigned long long tot = totals_host[c];
        const uint64_t s1 = tot >> shift, n1 = tot & ((1ull << shift) - 1);
        if (s1 > sink->kmer_cap || n1 > sink->id_cap || s1 < sink->kmers_done || n1 < sink->ids_done) break;
        const uint64_t s0 = sink->kmers_done, n0 = sink->ids_done;
        if (s1 > s0) {
            CU(cudaMemcpyAsync(sink->kmer_codes + s0 * KW, ctx->o_kmer_codes.as<uint64_t>() + s0 * KW, (s1 - s0) * KW * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->st_d2h));
            CU(cudaMemcpyAsync(sink->kmer_id_off + s0, ctx->o_kmer_id_off.as<uint64_t>() + s0, (s1 - s0) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->st_d2h));
        }
        if (n1 > n0) CU(cudaMemcpyAsync(sink->read_ids + n0, ctx->o_read_ids.as<int32_t>() + n0, (n1 - n0) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->st_d2h));
        sink->kmers_done = s1;
        sink->ids_done = n1;
    }
    return GBIN_OK;
}

// What was streamed into the sink belongs to an abandoned attempt: wait until nothing is in flight into the arenas, then start over.
int abandon_sink(gbin_ctx *ctx, HostSink *sink) {
    if (!sink) return GBIN_OK;
    CU(cudaStreamSynchronize(ctx->st_d2h));
    sink->kmers_done = sink->ids_done = 0;
    return GBIN_OK;
}

// Partition of n records by owner: launch(scratch, d_counts, st) runs the partition kernels and returns how many it launched.
template <typename Launch>
int partition_by_owner(gbin_ctx *ctx, uint64_t n, uint32_t n_parts, void *stream, uint64_t *counts_host, Launch launch) {
    if (!ctx || !counts_host || n_parts == 0 || n_parts > 256) return GBIN_E_INVALID_ARG;
    if (n >= (1ull << 32) - 8192) return fail(ctx, GBIN_E_TOO_LARGE, "too many records in one partition call");
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    CU(ctx->radix_scratch.ensure(radix_scratch_bytes(n)));
    const int launches = launch(ctx->radix_scratch.p, ctx->misc.as<Misc>()->part_counts, st);
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::part_counts, st));
    memcpy(counts_host, static_cast<Misc *>(ctx->h_misc.p)->part_counts, sizeof(uint64_t) * n_parts);
    ctx->tm.kernel_launches = (uint32_t)launches;
    return GBIN_OK;
}

__global__ void max_len_kernel(const uint32_t *__restrict__ lens, uint64_t n, unsigned int *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int v = i < n ? lens[i] : 0u;
    v = __reduce_max_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicMax(out, v);
}

struct WinCountIn {
    const uint32_t *c;
    __device__ __forceinline__ uint64_t operator()(uint64_t j) const { return c[j]; }
};

// Validates the reads descriptor (device pointers), finds max length and instance count.
// On return: *n_inst, *max_len, and for the ragged form ctx->rec_off holds per-read record offsets.
int plan_reads(gbin_ctx *ctx, const gbin_reads *rd, cudaStream_t st, uint64_t *n_inst, uint32_t *max_len, int *launches) {
    const int K = ctx->cfg.kmer_size;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    if (rd->n_reads == 0) {
        *n_inst = 0;
        *max_len = 0;
        return GBIN_OK;
    }
    if (!rd->data) return fail(ctx, GBIN_E_INVALID_ARG, "reads->data is NULL");
    if (rd->n_reads >= (1ull << 32)) return fail(ctx, GBIN_E_TOO_LARGE, "more than 2^32-1 reads in one batch");
    if (!rd->starts) {
        if (rd->stride < rd->read_len) return fail(ctx, GBIN_E_INVALID_ARG, "stride < read_len");
        if (rd->data_bytes && (rd->n_reads - 1) * rd->stride + rd->read_len > rd->data_bytes)
            return fail(ctx, GBIN_E_INVALID_ARG, "fixed-stride reads exceed data_bytes");
        *max_len = rd->read_len;
        *n_inst = rd->read_len >= (uint32_t)K ? rd->n_reads * (uint64_t)(rd->read_len - K + 1) : 0;
        return GBIN_OK;
    }
    if (!rd->lens) return fail(ctx, GBIN_E_INVALID_ARG, "ragged reads need lens");
    ReadsView rv{reinterpret_cast<const uint8_t *>(rd->data), rd->data_bytes, rd->n_reads, rd->stride, rd->read_len, rd->starts, rd->lens};
    CU(ctx->win_counts.ensure(rd->n_reads * sizeof(uint32_t)));
    CU(ctx->rec_off.ensure((rd->n_reads + 1) * sizeof(uint64_t)));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(rd->n_reads)));
    CU(cudaMemsetAsync(&dm->reads.max_len, 0, sizeof(unsigned int), st));
    if (rd->max_read_len == 0) {
        max_len_kernel<<<(unsigned)((rd->n_reads + 255) / 256), 256, 0, st>>>(rd->lens, rd->n_reads, &dm->reads.max_len);
        (*launches)++;
    }
    *launches += launch_count_windows(rv, K, ctx->win_counts.as<uint32_t>(), st);
    *launches += exclusive_scan<uint64_t, WinCountIn>(WinCountIn{ctx->win_counts.as<uint32_t>()}, ctx->rec_off.as<uint64_t>(), rd->n_reads,
                                                      ctx->scan_scratch.as<uint64_t>(),
                                                      reinterpret_cast<uint64_t *>(&dm->reads.total_windows), st);
    CU(read_back(ctx, &Misc::reads, st));
    *n_inst = hm->reads.total_windows;
    *max_len = rd->max_read_len ? rd->max_read_len : hm->reads.max_len;
    return GBIN_OK;
}

int run_scan(gbin_ctx *ctx, const gbin_reads *rd, uint32_t arrival_base, void *d_records, uint32_t max_len, cudaStream_t st, int *launches) {
    Misc *dm = ctx->misc.as<Misc>();
    ReadsView rv{reinterpret_cast<const uint8_t *>(rd->data), rd->data_bytes, rd->n_reads, rd->stride, rd->read_len, rd->starts, rd->lens};
    CU(cudaMemsetAsync(&dm->grp.bad_bases, 0, sizeof(unsigned long long), st));
    const bool on = ctx->prof.begin(KK_SCAN, st);
    const int ls = launch_scan_reads(rv, rd->starts ? ctx->rec_off.as<uint64_t>() : nullptr, ctx->cfg.kmer_size, ctx->cfg.mmer_size, ctx->KW,
                                     arrival_base, max_len ? max_len : 1, d_records, &dm->grp.bad_bases, ctx->sm_count, st);
    ctx->prof.end(on, ls < 0 ? 0 : ls, st);
    if (ls < 0) return fail(ctx, GBIN_E_TOO_LARGE, "a read of %u bases does not fit the scan kernel's shared memory (limit %u bases)", max_len, gbin_max_read_len());
    *launches += ls;
    CU(cudaGetLastError());
    return GBIN_OK;
}

// Sort + run-length + prune + emit of n records living in `recs` (scratch twin `twin`).
int run_group(gbin_ctx *ctx, void *recs, void *twin, uint64_t n, const int32_t *d_ids, int32_t id_base, cudaStream_t st,
              gbin_table *out, int *launches, cudaEvent_t ev_sorted) {
    const int KW = ctx->KW, K = ctx->cfg.kmer_size, M = ctx->cfg.mmer_size, cutoff = ctx->cfg.abundance_cutoff;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    CU(ctx->radix_scratch.ensure(radix_scratch_bytes(n)));
    bool in_b = false;
    int passes = 0;
    *launches += radix_sort_records(recs, twin, n, KW, K, M, ctx->radix_scratch.p, &in_b, &passes, &ctx->prof, st);
    CU(cudaGetLastError());
    ctx->tm.sort_passes = (uint32_t)passes;
    const void *sorted = in_b ? twin : recs;
    if (ev_sorted) CU(cudaEventRecord(ev_sorted, st));

    GroupWorkspace ws{};
    CU(ctx->group_of.ensure((n + 1) * sizeof(uint32_t)));
    CU(ctx->run_start.ensure((n + 2) * sizeof(uint32_t)));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n)));
    ws.group_of = ctx->group_of.as<uint32_t>();
    ws.run_start = ctx->run_start.as<uint32_t>();
    ws.scan_scratch = ctx->scan_scratch.p;
    ws.counts = &dm->grp.counts;
    ws.cutoff = cutoff;

    bool on = ctx->prof.begin(KK_RUNS, st);
    int lg = group_find_runs(sorted, n, KW, ws, st);
    ctx->prof.end(on, lg, st);
    *launches += lg;
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::grp, st));
    if (hm->grp.bad_bases) return fail(ctx, GBIN_E_NON_ACGT, "%llu bases other than A/C/G/T in the batch", hm->grp.bad_bases);
    const uint64_t G = hm->grp.counts.n_distinct;

    uint64_t S = 0, NS = 0, B = 0;
    if (G) {
        CU(ctx->surv_index.ensure((G + 1) * sizeof(uint32_t)));
        CU(ctx->id_offset.ensure((G + 1) * sizeof(uint64_t)));
        ws.surv_index = ctx->surv_index.as<uint32_t>();
        ws.id_offset = ctx->id_offset.as<uint64_t>();
        on = ctx->prof.begin(KK_PRUNE, st);
        lg = group_prune_offsets(n, G, cutoff, ws, st);
        ctx->prof.end(on, lg, st);
        *launches += lg;
        CU(cudaGetLastError());
        CU(read_back(ctx, &Misc::grp, st));
        S = hm->grp.counts.n_kmers;
        NS = hm->grp.counts.n_ids;
    }
    if (S) {
        CU(ctx->surv_group.ensure(S * sizeof(uint32_t)));
        CU(ctx->bucket_of.ensure(S * sizeof(uint32_t)));
        ws.surv_group = ctx->surv_group.as<uint32_t>();
        ws.bucket_of = ctx->bucket_of.as<uint32_t>();
        on = ctx->prof.begin(KK_PRUNE, st);
        lg = group_mark_buckets(sorted, KW, G, S, ws, st);
        ctx->prof.end(on, lg, st);
        *launches += lg;
        CU(cudaGetLastError());
        CU(read_back(ctx, &Misc::grp, st));
        B = hm->grp.counts.n_buckets;
    }
    CU(ctx->o_mmer_codes.ensure((B + 1) * sizeof(uint32_t)));
    CU(ctx->o_mmer_kmer_off.ensure((B + 1) * sizeof(uint64_t)));
    CU(ctx->o_kmer_codes.ensure((S * KW + 1) * sizeof(uint64_t)));
    CU(ctx->o_kmer_id_off.ensure((S + 1) * sizeof(uint64_t)));
    CU(ctx->o_read_ids.ensure((NS + 1) * sizeof(int32_t)));
    TableOut to{ctx->o_mmer_codes.as<uint32_t>(), ctx->o_mmer_kmer_off.as<uint64_t>(), ctx->o_kmer_codes.as<uint64_t>(),
                ctx->o_kmer_id_off.as<uint64_t>(), ctx->o_read_ids.as<int32_t>()};
    on = ctx->prof.begin(KK_EMIT, st);
    lg = group_emit(sorted, n, KW, G, S, NS, B, d_ids, id_base, ws, to, st);
    ctx->prof.end(on, lg, st);
    *launches += lg;
    CU(cudaGetLastError());
    *out = device_table(ctx, n, G, S, NS, B);
    return GBIN_OK;
}

// ---- super-k-mer pipelines.  Pipeline 2: super-k-mer records -> stable sort by m-mer -> grouping in shared memory.

// Scan stage of pipelines 2 and 3: one record per signature segment, in arrival order, into ctx->skr_a (own == true) or into the
// caller's buffer `ext` of `ext_cap` records.  *n_skr receives the record count.  With a feed (host path, fixed-stride
// reads) the reads arrive over PCIe in chunks on the copy stream and every chunk is scanned as soon as it is there.
int run_skr_scan(gbin_ctx *ctx, const gbin_reads *rd, uint64_t n, uint32_t max_len, uint32_t arrival_base, void *ext, uint64_t ext_cap,
                 cudaStream_t st, uint64_t *n_skr_out, int *launches, const HostFeed *feed = nullptr) {
    const int K = ctx->cfg.kmer_size, M = ctx->cfg.mmer_size;
    const int NW = K <= 32 ? 8 : 12;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    ReadsView rv{reinterpret_cast<const uint8_t *>(rd->data), rd->data_bytes, rd->n_reads, rd->stride, rd->read_len, rd->starts, rd->lens};
    uint64_t cap = ext ? ext_cap : n / 4 + rd->n_reads + 1024;
    if (!ext && cap > n) cap = n;
    uint64_t n_skr = 0;
    for (int attempt = 0; attempt < 2; attempt++) {
        if (!ext) CU(ctx->skr_a.ensure((cap + 1) * NW * 4));
        CU(ctx->tile_state.ensure((size_t)skr_scan_tiles(rd->n_reads, K, M, max_len) * 8 + 8));
        CU(cudaMemsetAsync(dm->skr_counters, 0, sizeof dm->skr_counters, st));
        const bool on = ctx->prof.begin(KK_SKR_SCAN, st);
        int ls = 0;
        const int chunks = (feed && attempt == 0) ? feed->chunks : 1;
        for (int c = 0; c < chunks; c++) {
            const uint64_t r0 = rd->n_reads * (uint64_t)c / chunks, r1 = rd->n_reads * (uint64_t)(c + 1) / chunks;
            if (feed && attempt == 0) {
                const uint64_t b0 = r0 * rd->stride, b1 = (c + 1 == chunks) ? feed->bytes : r1 * rd->stride;
                if (b1 > b0) CU(cudaMemcpyAsync(feed->dst + b0, feed->src + b0, b1 - b0, cudaMemcpyHostToDevice, ctx->st_h2d));
                CU(cudaEventRecord(ctx->ev_feed[c], ctx->st_h2d));
                CU(cudaStreamWaitEvent(st, ctx->ev_feed[c], 0));
                if (c + 1 == chunks) CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));  // every byte of the reads is on the device
            }
            const int l1 = launch_skr_scan(rv, r0, r1, K, M, arrival_base, max_len, ext ? ext : ctx->skr_a.p, cap, ctx->tile_state.as<unsigned long long>(),
                                           &dm->skr_ticket, dm->skr_counters, ctx->sm_count, st);
            if (l1 < 0) {  // reads too long for the shared memory of this kernel: the caller uses the instance-record scan
                if (feed && attempt == 0) CU(cudaStreamSynchronize(ctx->st_h2d));
                return GBIN_E_TOO_LARGE;
            }
            ls += l1;
        }
        ctx->prof.end(on, ls, st);
        *launches += ls;
        CU(cudaGetLastError());
        CU(read_back(ctx, &Misc::skr_counters, st));
        if (hm->skr_counters[0]) return fail(ctx, GBIN_E_NON_ACGT, "%llu bases other than A/C/G/T in the batch", hm->skr_counters[0]);
        n_skr = hm->skr_counters[1];
        if (hm->skr_counters[2] != n)
            return fail(ctx, GBIN_E_CUDA, "internal: scan produced %llu instances, expected %llu", hm->skr_counters[2], (unsigned long long)n);
        if (n_skr <= cap) break;
        if (ext) return fail(ctx, GBIN_E_INVALID_ARG, "super-k-mer buffer too small: need %llu records", (unsigned long long)n_skr);
        cap = n_skr;  // more segments than estimated: the kernel only counted; run it again with room for all
    }
    *n_skr_out = n_skr;
    return GBIN_OK;
}

// Sort + plan + group + emit over n_skr records in `skr` (clobbered; `twin` is the sort's second buffer).
// *done = false when a unit overflowed and the batch must go through pipeline v1.
int run_v2_group(gbin_ctx *ctx, void *skr, void *twin, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, gbin_table *out,
                 int *launches, bool *done, uint64_t *n_inst_out, HostSink *sink = nullptr) {
    *done = false;
    const int K = ctx->cfg.kmer_size, M = ctx->cfg.mmer_size, cutoff = ctx->cfg.abundance_cutoff, KW = ctx->KW;
    const int NW = K <= 32 ? 8 : 12;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);

    // ---- level 1: stable sort of the records by m-mer code
    CU(ctx->radix_scratch.ensure(radix_scratch_bytes(n_skr)));
    bool in_b = false;
    int passes = 0;
    CU(ctx->skr_side.ensure((n_skr + 2) * 8));
    *launches += radix_sort_skr_by_mmer(skr, twin, n_skr, NW, M, ctx->radix_scratch.p, &in_b, &passes, ctx->skr_side.as<uint64_t>(), &ctx->prof, st);
    CU(cudaGetLastError());
    ctx->tm.sort_passes = (uint32_t)passes;
    const void *sorted = in_b ? twin : skr;
    CU(cudaEventRecord(ctx->ev[EV_SORTED], st));

    // ---- plan: instance prefix, m-mer runs, units
    CU(ctx->inst_prefix.ensure((n_skr + 2) * 4));
    CU(ctx->run_excl.ensure((n_skr + 2) * 8));
    CU(ctx->skr_run_start.ensure((n_skr + 2) * 4));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n_skr)));
    bool on = ctx->prof.begin(KK_SKR_PLAN, st);
    int lp = skr_plan_runs(ctx->skr_side.as<uint64_t>(), n_skr, ctx->inst_prefix.as<uint32_t>(), ctx->run_excl.as<uint64_t>(), ctx->skr_run_start.as<uint32_t>(),
                           ctx->scan_scratch.as<uint64_t>(), &dm->plan.n_inst, &dm->plan.n_runs, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::plan, st));
    const uint64_t n_runs = hm->plan.n_runs, n = hm->plan.n_inst;
    *n_inst_out = n;
    ctx->rs.n_super_kmers = n_skr;
    ctx->rs.n_mmer_runs = n_runs;
    const uint64_t max_units = skr_max_units(n, n_runs);
    CU(ctx->small_prefix.ensure((n_runs + 1) * 4));
    CU(ctx->unit_base.ensure((n_runs + 1) * 4));
    CU(ctx->units.ensure(max_units * skr_unit_bytes()));
    CU(ctx->unit_state.ensure(max_units * 8));
    CU(ctx->big_list.ensure(skr_max_big_runs(n) * 8));
    CU(ctx->big_k0.ensure((n + 1) * 8));
    if (KW == 2) CU(ctx->big_k1.ensure((n + 1) * 8));
    CU(ctx->big_arr.ensure((n + 1) * 4));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n / 2 + n_runs + 1024)));
    on = ctx->prof.begin(KK_SKR_PLAN, st);
    lp = skr_plan_units(sorted, K, ctx->inst_prefix.as<uint32_t>(), ctx->skr_run_start.as<uint32_t>(), n_runs, ctx->small_prefix.as<uint32_t>(),
                        ctx->unit_base.as<uint32_t>(), ctx->scan_scratch.as<uint32_t>(), ctx->units.p, max_units, &dm->gc, ctx->big_list.as<uint32_t>(),
                        ctx->big_k0.as<uint64_t>(), ctx->big_k1.as<uint64_t>(), ctx->big_arr.as<uint32_t>(), ctx->sm_count, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());

    // ---- level 2 + prune + emit. Output bounds: a surviving k-mer has more than `cutoff` instances.
    const uint64_t kmer_cap = cutoff >= 0 ? n / ((uint64_t)cutoff + 1) + 1 : n + 1;
    CU(ctx->o_kmer_codes.ensure((kmer_cap * KW + 1) * sizeof(uint64_t)));
    CU(ctx->o_kmer_mmer.ensure((kmer_cap + 1) * sizeof(uint32_t)));
    CU(ctx->o_kmer_id_off.ensure((kmer_cap + 2) * sizeof(uint64_t)));
    CU(ctx->o_read_ids.ensure((n + 1) * sizeof(int32_t)));
    CU(ctx->stg_ids.ensure((n + 1) * sizeof(int32_t)));
    CU(ctx->stg_codes.ensure((kmer_cap * KW + 1) * sizeof(uint64_t)));
    CU(ctx->stg_mmer.ensure((kmer_cap + 1) * sizeof(uint32_t)));
    CU(ctx->stg_off.ensure((kmer_cap + 1) * sizeof(uint32_t)));
    on = ctx->prof.begin(KK_SKR_GROUP, st);
    SkrGroupChunks ch{1u, dm->chunk_tickets, nullptr, nullptr, nullptr};
    if (sink && sink->chunks > 1) {
        ch.n = (uint32_t)sink->chunks;
        ch.totals_dev = dm->chunk_totals;
        ch.totals_host = hm->chunk_totals;
        ch.done = ctx->ev_chunk;
    }
    lp = skr_group_launch(sorted, K, cutoff, ctx->inst_prefix.as<uint32_t>(), ctx->units.p, ctx->unit_state.as<unsigned long long>(), max_units, ch,
                          &dm->gc, ctx->big_k0.as<uint64_t>(), ctx->big_k1.as<uint64_t>(), ctx->big_arr.as<uint32_t>(), d_ids, id_base, ctx->o_kmer_codes.as<uint64_t>(), ctx->o_kmer_mmer.as<uint32_t>(),
                          ctx->o_kmer_id_off.as<uint64_t>(), ctx->o_read_ids.as<int32_t>(), kmer_cap, n, ctx->stg_ids.as<int32_t>(), ctx->stg_codes.as<uint64_t>(),
                          ctx->stg_mmer.as<uint32_t>(), ctx->stg_off.as<uint32_t>(), ctx->sm_count, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    if (ch.done) {  // the grouping kernels pack each chunk's totals as {k-mers << 31 | ids}
        const int rc = stream_finished_chunks(ctx, sink, ch.n, hm->chunk_totals, 31, nullptr);
        if (rc) return rc;
    }
    CU(read_back(ctx, &Misc::gc, st));
    ctx->rs.n_units = hm->gc.n_units;
    if (hm->gc.overflow) {  // a unit did not fit shared memory: this batch goes through pipeline v1
        ctx->fallbacks++;
        return GBIN_OK;
    }
    const uint64_t S = hm->gc.total_kmers, NS = hm->gc.total_ids;
    uint64_t B = 0;
    const int rc = emit_bucket_directory(ctx, S, NS, st, launches, &B);
    if (rc) return rc;
    *out = device_table(ctx, n, hm->gc.distinct, S, NS, B);
    *done = true;
    return GBIN_OK;
}

// ---- pipeline 3: entries sorted by reference, one warp (512-instance units) or one pair of warps (1024-instance units) per unit,
// staging + finalize (bin3.cu)
// The records in `skr` are read, not moved.  *done = false when the batch does not fit (a (bucket, d) class larger than a unit);
// it then goes through pipeline 2, which sorts the records themselves.

// Key layout for this batch: explicit (gbin_set_tuning v3_nc = 1 | 2) or chosen from the mean m-mer bucket size (v3_nc = 0):
// buckets that fit a unit need nothing but the m-mer code; larger ones are broken up by extending the key (bin3.cuh).
int v3_choose_layout(gbin_ctx *ctx, const void *skr, uint64_t n_skr, cudaStream_t st, KeyLayout *out, int *launches) {
    const int K = ctx->cfg.kmer_size, M = ctx->cfg.mmer_size;
    // Unit capacity: 1024 instances when whole m-mer buckets are units (fewer buckets straddle units), 512 when the key is
    // extended or the k-mers are two words wide (twice the warps per SM: the grouping kernel is latency-bound; measured
    // 17.1 -> 11.3 ms on a config-3 shaped batch, 13.4 -> 7.9 ms on a config-5 shaped one).
    auto set_cap = [&](const KeyLayout &kl) { ctx->v3_cap_eff = ctx->v3_cap ? ctx->v3_cap : ((ctx->KW == 2 || kl.nc == 2) ? 512 : 1024); };
    if (ctx->v3_nc != 0) {
        *out = make_key_layout(K, M, ctx->v3_h, ctx->v3_nc);
        set_cap(*out);
        return GBIN_OK;
    }
    if (2 * M + 2 > 31 || M > 13 || n_skr == 0) {  // no room for a longer key / code space too large for the bitmap: plain m-mer keys
        *out = make_key_layout(K, M, 0, 1);
        set_cap(*out);
        return GBIN_OK;
    }
    // the decision is kept for batches of similar size on this context
    if (ctx->v3_auto_n && n_skr >= ctx->v3_auto_n / 2 && n_skr <= ctx->v3_auto_n * 2) {
        *out = make_key_layout(K, M, ctx->v3_auto_h, ctx->v3_auto_nc);
        set_cap(*out);
        return GBIN_OK;
    }
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    CU(ctx->v3_bitmap.ensure(v3_mmer_bitmap_bytes(M)));
    *launches += v3_count_mmers(skr, K <= 32 ? 8 : 12, n_skr, M, ctx->v3_bitmap.as<uint32_t>(), &dm->n_mmers, st);
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::n_mmers, st));
    const double buckets = hm->n_mmers ? (double)hm->n_mmers : 1.0;
    const double mean_inst = (double)n_skr / buckets * ((K - M + 2) / 2.0);  // a record holds about (K-M+2)/2 windows
    int nc = 1, h = 0;
    const int cap1 = ctx->v3_cap ? ctx->v3_cap : 1024, cap2 = ctx->v3_cap ? ctx->v3_cap : 512;
    if (mean_inst > cap1 / 2.5) {
        nc = 2;
        double per = mean_inst / 2.0;
        while (per > cap2 / 8.0 && h < 15) {
            per /= 4.0;
            h++;
        }
    }
    *out = make_key_layout(K, M, h, nc);
    set_cap(*out);
    ctx->v3_auto_n = n_skr;
    ctx->v3_auto_h = out->h;
    ctx->v3_auto_nc = out->nc;
    return GBIN_OK;
}

// One pass of pipeline 3 over the sorted entries [ent, ent + n_ent): plan, group, finalize; the pass's k-mers / ids are appended to
// the table behind the S_off k-mers / N_off ids of the passes before it.  *ok = false: the pass does not fit (see run_v3_group).
int run_v3_pass(gbin_ctx *ctx, const void *skr, const uint64_t *ent, const uint16_t *sorted_info, uint64_t n_ent, const KeyLayout &kl, const int32_t *d_ids, int32_t id_base, cudaStream_t st,
                uint64_t S_off, uint64_t N_off, bool single_pass, HostSink *sink, int *launches, bool *ok, uint64_t *n_inst, uint64_t *distinct, uint64_t *S_out,
                uint64_t *N_out) {
    *ok = false;
    const int cutoff = ctx->cfg.abundance_cutoff, KW = ctx->KW;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    // ---- plan: instance prefix, atoms, units
    CU(ctx->inst_prefix.ensure((n_ent + 2) * 4));
    CU(ctx->run_excl.ensure((n_ent + 2) * 8));
    CU(ctx->skr_run_start.ensure((n_ent + 2) * 4));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n_ent)));
    bool on = ctx->prof.begin(KK_SKR_PLAN, st);
    int lp = v3_plan_runs(ent, sorted_info, n_ent, ctx->inst_prefix.as<uint32_t>(), ctx->run_excl.as<uint64_t>(), ctx->skr_run_start.as<uint32_t>(),
                          ctx->scan_scratch.as<uint64_t>(), &dm->plan.n_inst, &dm->plan.n_runs, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::plan, st));
    const uint64_t n_runs = hm->plan.n_runs, n = hm->plan.n_inst;
    *n_inst = n;
    ctx->rs.n_mmer_runs += n_runs;
    const uint64_t max_units = v3_max_units(n, n_runs, ctx->v3_cap_eff);
    CU(ctx->small_prefix.ensure((n_runs + 2) * 8));
    CU(ctx->v3_base64.ensure((n_runs + 2) * 8));
    CU(ctx->v3_atoms.ensure((4 * n_runs + 8) * 4));
    CU(ctx->v3_head_run.ensure((max_units + 1) * 4));
    CU(ctx->units.ensure(max_units * v3_unit_bytes()));
    CU(ctx->v3_unit_out.ensure(max_units * v3_unit_out_bytes()));
    CU(ctx->v3_unit_excl.ensure((2 * max_units + 2) * 8));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n_runs + max_units + 1024)));
    V3Chunks ch{1u, dm->v3_tickets, dm->chunk_bounds, &dm->v3_chunk_sum, dm->chunk_totals, dm->lsd_totals, nullptr, nullptr, nullptr,
                ctx->st_aux, ctx->ev_fork, ctx->ev_join};
    if (single_pass && sink && sink->chunks > 1) {
        ch.n = (uint32_t)sink->chunks;
        ch.totals_host = hm->chunk_totals;
        ch.lsd_totals_host = hm->lsd_totals;
        ch.done = ctx->ev_chunk;
    }
    on = ctx->prof.begin(KK_SKR_PLAN, st);
    lp = v3_plan_units(sorted_info, ent, kl, ctx->v3_cap_eff, ctx->inst_prefix.as<uint32_t>(), ctx->skr_run_start.as<uint32_t>(), n_runs, ctx->small_prefix.as<uint64_t>(),
                       ctx->v3_base64.as<uint64_t>(), ctx->v3_atoms.as<uint32_t>(), ctx->v3_atoms.as<uint32_t>() + 3 * n_runs, ctx->v3_head_run.as<uint32_t>(),
                       ctx->scan_scratch.p, ctx->units.p, max_units, &dm->gc3, ch.n, dm->chunk_bounds, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());

    // ---- level 2 + prune + emit.  Output bounds: a surviving k-mer has more than `cutoff` instances.
    const uint64_t kmer_cap = cutoff >= 0 ? n / ((uint64_t)cutoff + 1) + 1 : n + 1;
    CU(ctx->o_kmer_codes.ensure_keep(((S_off + kmer_cap) * KW + 1) * sizeof(uint64_t), S_off * KW * sizeof(uint64_t), st));
    CU(ctx->o_kmer_mmer.ensure_keep((S_off + kmer_cap + 1) * sizeof(uint32_t), S_off * sizeof(uint32_t), st));
    CU(ctx->o_kmer_id_off.ensure_keep((S_off + kmer_cap + 2) * sizeof(uint64_t), S_off * sizeof(uint64_t), st));
    CU(ctx->o_read_ids.ensure_keep((N_off + n + 1) * sizeof(int32_t), N_off * sizeof(int32_t), st));
    CU(ctx->stg_ids.ensure((n + 1) * sizeof(int32_t)));
    CU(ctx->stg_codes.ensure((kmer_cap * KW + 1) * sizeof(uint64_t)));
    CU(ctx->stg_mmer.ensure((kmer_cap + 1) * sizeof(uint32_t)));
    CU(ctx->stg_off.ensure((kmer_cap + 1) * sizeof(uint32_t)));
    V3Out vo{ctx->o_kmer_codes.as<uint64_t>() + S_off * KW, ctx->o_kmer_mmer.as<uint32_t>() + S_off, ctx->o_kmer_id_off.as<uint64_t>() + S_off,
             ctx->o_read_ids.as<int32_t>() + N_off, kmer_cap, n, ctx->stg_codes.as<uint64_t>(), ctx->stg_mmer.as<uint32_t>(), ctx->stg_off.as<uint32_t>(),
             ctx->stg_ids.as<int32_t>(), ctx->v3_unit_out.p, N_off};
    const size_t rb = sizeof(uint64_t) * KW + 8;
    auto lsd_arrays = [&](uint64_t cap) -> int {  // arrays of the global sort for long spans, for `cap` k-mers
        if (cap == 0) return GBIN_OK;
        CU(ctx->rec_a.ensure((cap + 1) * rb));
        CU(ctx->rec_b.ensure((cap + 1) * rb));
        CU(ctx->v3_lsd_aux.ensure((cap + 1) * 16));
        return GBIN_OK;
    };
    // long spans appear when buckets are large enough for extended keys; their k-mers are a fraction of the bound (grown on demand)
    uint64_t lsd_cap = (kl.nc == 2 || ctx->v3_lsd_seen) ? (kmer_cap < (1u << 22) ? kmer_cap : kmer_cap / 4) : 0;
    if (lsd_cap && lsd_cap < ctx->v3_lsd_cap_seen && ctx->v3_lsd_cap_seen <= kmer_cap) lsd_cap = ctx->v3_lsd_cap_seen;
    int rc = lsd_arrays(lsd_cap);
    if (rc) return rc;
    auto lsd_view = [&](uint64_t cap) {
        uint32_t *aux = ctx->v3_lsd_aux.as<uint32_t>();
        return cap ? V3Lsd{ctx->rec_a.p, aux, aux + (cap + 1), aux + 2 * (cap + 1), aux + 3 * (cap + 1), cap} : V3Lsd{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    };
    uint64_t *unit_excl = ctx->v3_unit_excl.as<uint64_t>(), *lsd_excl = unit_excl + max_units + 1;
    lp = v3_group_launch(skr, ent, ctx->units.p, kl, ctx->v3_cap_eff, cutoff, d_ids, id_base, vo, max_units, unit_excl, lsd_excl, ctx->scan_scratch.p, &dm->gc3, ch,
                         lsd_view(lsd_cap), false, ctx->sm_count, &ctx->prof, st);
    *launches += lp;
    CU(cudaGetLastError());
    if (ch.done) {  // the grouping kernels pack each chunk's totals as {k-mers << 32 | ids}
        rc = stream_finished_chunks(ctx, sink, ch.n, hm->chunk_totals, 32, hm->lsd_totals);
        if (rc) return rc;
    }
    CU(read_back(ctx, &Misc::gc3, st));
    if (hm->gc3.overflow == 6u && hm->gc3.lsd_kmers > lsd_cap) {
        // long spans met no (or too small) sort arrays: allocate them and redo their placement (the staged results are still there)
        ctx->v3_lsd_seen = true;
        lsd_cap = hm->gc3.lsd_kmers + hm->gc3.lsd_kmers / 16 + 1024;
        if (lsd_cap > kmer_cap) lsd_cap = kmer_cap;
        ctx->v3_lsd_cap_seen = lsd_cap;
        rc = lsd_arrays(lsd_cap);
        if (rc) return rc;
        CU(cudaMemsetAsync(&dm->gc3.overflow, 0, sizeof(unsigned int), st));
        V3Chunks ch1 = ch;
        ch1.totals_host = ch1.lsd_totals_host = nullptr;
        ch1.done = nullptr;
        lp = v3_group_launch(skr, ent, ctx->units.p, kl, ctx->v3_cap_eff, cutoff, d_ids, id_base, vo, max_units, unit_excl, lsd_excl, ctx->scan_scratch.p, &dm->gc3, ch1,
                             lsd_view(lsd_cap), true, ctx->sm_count, &ctx->prof, st);
        *launches += lp;
        CU(cudaGetLastError());
        CU(read_back(ctx, &Misc::gc3, st));
    }
    ctx->rs.n_units += hm->gc3.n_units;
    ctx->rs.n_lsd_kmers += hm->gc3.lsd_kmers;
    if (hm->gc3.overflow) {  // not done: the caller falls back
        snprintf(ctx->err, sizeof ctx->err, "pipeline 3 gave the batch up (code %u: a (bucket, d) class larger than a unit)", hm->gc3.overflow);
        return GBIN_OK;
    }
    if (hm->gc3.lsd_kmers) {
        const uint64_t nl = hm->gc3.lsd_kmers;
        CU(ctx->radix_scratch.ensure(radix_scratch_bytes(nl)));
        CU(ctx->run_excl.ensure((nl + 2) * 8));
        CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(nl + 1024)));
        lp = v3_lsd_finish(kl, nl, ctx->rec_a.p, ctx->rec_b.p, ctx->radix_scratch.p, ctx->run_excl.as<uint64_t>(), ctx->scan_scratch.p, vo, lsd_view(lsd_cap), ctx->sm_count, &ctx->prof,
                           st);
        *launches += lp;
        CU(cudaGetLastError());
    }
    *distinct = hm->gc3.distinct;
    *S_out = hm->gc3.total_kmers;
    *N_out = hm->gc3.total_ids;
    *ok = true;
    return GBIN_OK;
}

int run_v3_group(gbin_ctx *ctx, const void *skr, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, gbin_table *out, int *launches,
                 bool *done, uint64_t *n_inst_out, HostSink *sink = nullptr) {
    *done = false;
    const int K = ctx->cfg.kmer_size, M = ctx->cfg.mmer_size;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    KeyLayout kl;
    int rc = v3_choose_layout(ctx, skr, n_skr, st, &kl, launches);
    if (rc) return rc;
    if (n_skr >= (1ull << (32 - kl.cshift))) return GBIN_OK;  // slots are 32-bit
    memset(&ctx->rs, 0, sizeof ctx->rs);
    ctx->rs.n_super_kmers = n_skr;
    ctx->rs.key_nc = (uint32_t)kl.nc;
    ctx->rs.key_h = (uint32_t)kl.h;

    // ---- entries + level 1: stable sort of the entries by key
    const uint64_t n_slots = n_skr << kl.cshift;
    // the two entry buffers of the sort: in donated memory when the caller gave enough of it (the multi-GPU path hands over the
    // scan's record buffer, dead after the exchange — one allocation of that size less per step), else the context's own
    const uint64_t ent_bytes = ((n_slots + 2) * 8 + 255) & ~255ull;
    uint64_t *ent_a_p, *ent_b_p;
    if (ctx->donated && ctx->donated_bytes >= 2 * ent_bytes && (reinterpret_cast<uintptr_t>(ctx->donated) & 15u) == 0) {
        ent_a_p = static_cast<uint64_t *>(ctx->donated);
        ent_b_p = ent_a_p + ent_bytes / 8;
        if (ctx->ent_a.cap + ctx->ent_b.cap > (1ull << 30)) {  // a large batch on donated memory: the own buffers of an earlier one would only crowd the HBM
            ctx->ent_a.release();
            ctx->ent_b.release();
        }
    } else {
        CU(ctx->ent_a.ensure(ent_bytes));
        CU(ctx->ent_b.ensure(ent_bytes));
        ent_a_p = ctx->ent_a.as<uint64_t>();
        ent_b_p = ctx->ent_b.as<uint64_t>();
    }
    ctx->donated = nullptr;  // one call only
    ctx->donated_bytes = 0;
    CU(ctx->piece_n.ensure((n_slots + 16) * 2));
    CU(ctx->sorted_info.ensure((n_slots + 16) * 2));
    bool on = ctx->prof.begin(KK_V3_ENTRIES, st);
    int lp = v3_make_entries(skr, n_skr, kl, ent_a_p, ctx->piece_n.as<uint16_t>(), &dm->n_real_entries, st);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    CU(ctx->radix_scratch.ensure(radix_scratch_bytes(n_slots)));
    bool in_b = false;
    int passes = 0;
    *launches += radix_sort_entries(ent_a_p, ent_b_p, n_slots, kl.key_bits, ctx->radix_scratch.p, &in_b, &passes, ctx->piece_n.as<uint16_t>(),
                                    ctx->sorted_info.as<uint16_t>(), &ctx->prof, st, kl.nc == 2 ? &dm->n_real_entries : nullptr);
    CU(cudaGetLastError());
    ctx->tm.sort_passes = (uint32_t)passes;
    const uint64_t *ent = in_b ? ent_b_p : ent_a_p;
    CU(cudaEventRecord(ctx->ev[EV_SORTED], st));
    uint64_t n_ent = n_slots;
    if (kl.nc == 2) {  // empty pieces carry the all-ones key and sort behind everything: plan over the real ones only
        CU(read_back(ctx, &Misc::n_real_entries, st));
        n_ent = hm->n_real_entries;
    }

    // ---- passes: ranges of the sorted entries with at most pass_max k-mer instances each, cut between m-mer buckets
    std::vector<uint64_t> bounds{0, n_ent};
    const uint64_t pass_max = ctx->v3_pass_max;
    if (n_skr * (uint64_t)(K - M + 1) > pass_max) {  // more than one pass is possible: look at the instance counts
        const uint32_t nt = v3_pass_tiles(n_ent);
        CU(ctx->scan_scratch.ensure((size_t)nt * 8 + 64));
        unsigned long long *sums_dev = ctx->scan_scratch.as<unsigned long long>();
        *launches += v3_pass_tile_sums(ctx->sorted_info.as<uint16_t>(), n_ent, sums_dev, st);
        std::vector<unsigned long long> sums(nt);
        CU(cudaMemcpyAsync(sums.data(), sums_dev, (size_t)nt * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        std::vector<unsigned long long> cuts;
        unsigned long long acc = 0, all = 0;
        for (uint32_t t = 0; t < nt; t++) all += sums[t];
        // a batch of several passes is a batch that crowds the HBM: the workspace of a pass (staging, bounds of the table's growth) scales
        // with the pass, so such a batch is cut into passes of half the size
        const uint64_t pass_max = all > 2 * ctx->v3_pass_max ? ctx->v3_pass_max / 2 : ctx->v3_pass_max;
        for (uint32_t t = 0; t < nt; t++) {
            if (acc && acc + sums[t] > pass_max) {
                cuts.push_back((unsigned long long)t * v3_pass_tile_entries());
                acc = 0;
            }
            acc += sums[t];
        }
        if (!cuts.empty()) {
            CU(cudaMemcpyAsync(sums_dev, cuts.data(), cuts.size() * 8, cudaMemcpyHostToDevice, st));
            *launches += v3_pass_bounds(ent, n_ent, kl.mshift, sums_dev, (uint32_t)cuts.size(), st);
            CU(cudaMemcpyAsync(cuts.data(), sums_dev, cuts.size() * 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            bounds.assign(1, 0);
            for (unsigned long long c : cuts)
                if (c > bounds.back() && c < n_ent) bounds.push_back(c);
            bounds.push_back(n_ent);
        }
    }
    const bool single = bounds.size() == 2;
    uint64_t S_off = 0, N_off = 0, n_total = 0, distinct = 0;
    for (size_t p = 0; p + 1 < bounds.size(); p++) {
        bool ok = false;
        uint64_t n_p = 0, d_p = 0, S_p = 0, N_p = 0;
        rc = run_v3_pass(ctx, skr, ent + bounds[p], ctx->sorted_info.as<uint16_t>() + bounds[p], bounds[p + 1] - bounds[p], kl, d_ids, id_base, st, S_off, N_off, single, sink, launches, &ok, &n_p, &d_p, &S_p, &N_p);
        if (rc) return rc;
        if (!ok) return GBIN_OK;  // not done: the caller falls back
        S_off += S_p;
        N_off += N_p;
        n_total += n_p;
        distinct += d_p;
    }
    *n_inst_out = n_total;
    ctx->rs.n_passes = (uint32_t)(bounds.size() - 1);
    const uint64_t S = S_off, NS = N_off;
    if (S >= (1ull << 32)) return fail(ctx, GBIN_E_TOO_LARGE, "%llu surviving k-mers in one batch (limit 2^32)", (unsigned long long)S);
    uint64_t B = 0;
    rc = emit_bucket_directory(ctx, S, NS, st, launches, &B);
    if (rc) return rc;
    *out = device_table(ctx, n_total, distinct, S, NS, B);
    *done = true;
    return GBIN_OK;
}

// Group stage of the super-k-mer pipelines: v3 first (when configured), then v2.  *used receives the pipeline that made the table.
int run_skr_group(gbin_ctx *ctx, void *skr, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, gbin_table *out, int *launches, bool *done,
                  uint64_t *n_inst_out, HostSink *sink, int *used) {
    *done = false;
    const int NW = ctx->cfg.kmer_size <= 32 ? 8 : 12;
    if (ctx->pipeline >= 3) {
        int rc = run_v3_group(ctx, skr, n_skr, d_ids, id_base, st, out, launches, done, n_inst_out, sink);
        if (rc) return rc;
        if (*done) {
            *used = 3;
            return GBIN_OK;
        }
        ctx->fallbacks++;
        rc = abandon_sink(ctx, sink);
        if (rc) return rc;
    }
    if (n_skr * (uint64_t)(ctx->cfg.kmer_size - ctx->cfg.mmer_size + 1) >= (1ull << 31))  // pipeline 2 holds instance coordinates in 31 bits
        return fail(ctx, GBIN_E_TOO_LARGE, "the batch is too large for pipeline 2 (%llu super-k-mer records) and pipeline 3 %s", (unsigned long long)n_skr,
                    ctx->pipeline >= 3 ? "gave it up" : "is switched off");
    CU(ctx->skr_b.ensure((n_skr + 1) * NW * 4));
    int rc = run_v2_group(ctx, skr, ctx->skr_b.p, n_skr, d_ids, id_base, st, out, launches, done, n_inst_out, sink);
    if (rc) return rc;
    if (*done) *used = 2;
    return GBIN_OK;
}

int run_skr_pipelines(gbin_ctx *ctx, const gbin_reads *rd, uint64_t n, uint32_t max_len, cudaStream_t st, gbin_table *out, int *launches, bool *done,
                      const HostFeed *feed, HostSink *sink, int *used) {
    *done = false;
    if (n == 0 || (ctx->pipeline < 3 && n >= (1ull << 31))) return GBIN_OK;
    uint64_t n_skr = 0, n_chk = 0;
    int rc = run_skr_scan(ctx, rd, n, max_len, 0, nullptr, 0, st, &n_skr, launches, feed);
    if (rc == GBIN_E_TOO_LARGE) {  // reads longer than the super-k-mer scan holds in shared memory: pipeline 1 takes the batch
        ctx->fallbacks++;
        return GBIN_OK;
    }
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_SCANNED], st));
    rc = run_skr_group(ctx, ctx->skr_a.p, n_skr, rd->read_ids, rd->id_base, st, out, launches, done, &n_chk, sink, used);
    if (rc) return rc;
    if (!*done) return GBIN_OK;
    if (n_chk != n) return fail(ctx, GBIN_E_CUDA, "internal: record windows sum to %llu, expected %llu", (unsigned long long)n_chk, (unsigned long long)n);
    return GBIN_OK;
}

// feed: the reads have NOT been copied to rd->data yet (host path); whoever consumes them first issues the copy.
int bin_device_impl(gbin_ctx *ctx, const gbin_reads *rd, cudaStream_t st, gbin_table *out, int *launches, const HostFeed *feed = nullptr,
                    HostSink *sink = nullptr) {
    uint64_t n = 0;
    uint32_t max_len = 0;
    int rc = plan_reads(ctx, rd, st, &n, &max_len, launches);
    if (rc) return rc;
    if (max_len > gbin_max_read_len()) return fail(ctx, GBIN_E_TOO_LARGE, "read length %u exceeds the limit of %u bases", max_len, gbin_max_read_len());
    if (ctx->pipeline < 3 && n >= (1ull << 32) - 8192)
        return fail(ctx, GBIN_E_TOO_LARGE, "%llu k-mer instances in one batch (pipelines 1 and 2 hold 2^32; pipeline 3 works in passes)", (unsigned long long)n);
    const bool v2 = ctx->pipeline >= 2 && n != 0 && (ctx->pipeline >= 3 || n < (1ull << 31));
    if (feed && (!v2 || max_len > 1500)) {  // nobody downstream streams the reads in (long reads go to pipeline 1's scan): copy them in one piece
        CU(cudaMemcpyAsync(feed->dst, feed->src, feed->bytes, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
        feed = nullptr;
    }
    if (v2) {
        bool done = false;
        int used = 2;
        rc = run_skr_pipelines(ctx, rd, n, max_len, st, out, launches, &done, feed, sink, &used);
        if (rc) return rc;
        if (done) {
            ctx->last_pipeline = used;
            CU(cudaEventRecord(ctx->ev[EV_GROUPED], st));
            return GBIN_OK;
        }
        rc = abandon_sink(ctx, sink);
        if (rc) return rc;
    }
    if (n >= (1ull << 32) - 8192) return fail(ctx, GBIN_E_TOO_LARGE, "%llu k-mer instances: too many for the pipeline-1 fallback", (unsigned long long)n);
    ctx->last_pipeline = 1;
    memset(&ctx->rs, 0, sizeof ctx->rs);
    const size_t rb = sizeof(uint64_t) * ctx->KW + 8;
    CU(ctx->rec_a.ensure((n + 1) * rb));
    CU(ctx->rec_b.ensure((n + 1) * rb));
    rc = run_scan(ctx, rd, 0, ctx->rec_a.p, max_len, st, launches);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_SCANNED], st));
    rc = run_group(ctx, ctx->rec_a.p, ctx->rec_b.p, n, rd->read_ids, rd->id_base, st, out, launches, ctx->ev[EV_SORTED]);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_GROUPED], st));
    return GBIN_OK;
}

}  // namespace

extern "C" {

const char *gbin_strerror(int code) {
    switch (code) {
        case GBIN_OK: return "ok";
        case GBIN_E_INVALID_CONFIG: return "unsupported K/M (need 2 <= M <= 15 and 2M <= K <= 64)";
        case GBIN_E_CUDA: return "CUDA error";
        case GBIN_E_NOMEM: return "out of memory";
        case GBIN_E_NON_ACGT: return "read contains a byte other than A/C/G/T";
        case GBIN_E_STATE: return "call sequence error";
        case GBIN_E_TOO_LARGE: return "batch exceeds an implementation limit";
        case GBIN_E_INVALID_ARG: return "invalid argument";
        case GBIN_E_IO: return "I/O error";
        default: return "unknown error";
    }
}

const char *gbin_last_error(const gbin_ctx *ctx) { return ctx ? ctx->err : ""; }
int gbin_version(void) { return 100; }

int gbin_create(const gbin_config *cfg, gbin_ctx **out) {
    if (!out) return GBIN_E_INVALID_ARG;
    *out = nullptr;
    int rc = check_config(cfg);
    if (rc) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        return GBIN_E_CUDA;  // no CPU fallback: without a CUDA device the library refuses to work
    }
    if (cfg->device < 0 || cfg->device >= ndev) return GBIN_E_INVALID_ARG;
    gbin_ctx *ctx = new (std::nothrow) gbin_ctx();
    if (!ctx) return GBIN_E_NOMEM;
    ctx->cfg = *cfg;
    ctx->KW = cfg->kmer_size <= 32 ? 1 : 2;
    ctx->err[0] = 0;
    ctx->pipeline = 3;
    if (const char *e = getenv("GBIN_PIPELINE")) {
        const int v = atoi(e);
        ctx->pipeline = (v >= 1 && v <= 3) ? v : 3;
    }
    ctx->v3_h = 0;
    ctx->v3_nc = 0;  // automatic
    if (const char *e = getenv("GBIN_V3_NC")) {
        const int v = atoi(e);
        ctx->v3_nc = (v == 1 || v == 2) ? v : 0;
    }
    if (const char *e = getenv("GBIN_V3_H")) ctx->v3_h = atoi(e);
    if (const char *e = getenv("GBIN_V3_PASS_MAX")) {
        const long long v = atoll(e);
        if (v >= 1000) ctx->v3_pass_max = (uint64_t)v;
    }
    // 128-bit k-mer codes double the shared memory of a unit: units of 512 instances keep the warps per SM up
    ctx->v3_cap = 0;
    ctx->v3_cap_eff = ctx->KW == 2 ? 512 : 1024;
    if (const char *e = getenv("GBIN_XCHG_TIMEOUT_MS"))
        if (atoi(e) >= 100) ctx->xchg_timeout_ms = atoi(e);
    if (const char *e = getenv("GBIN_V3_CAP")) ctx->v3_cap = atoi(e) == 512 ? 512 : (atoi(e) == 1024 ? 1024 : 0);
    ctx->last_pipeline = 0;
    ctx->fallbacks = 0;
    memset(&ctx->rs, 0, sizeof ctx->rs);
    memset(&ctx->tm, 0, sizeof ctx->tm);
    ctx->prof.reset();
    cudaError_t e = cudaSetDevice(cfg->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->st_h2d, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->st_d2h, cudaStreamNonBlocking);
    for (int i = 0; i < EV_COUNT && e == cudaSuccess; i++) e = cudaEventCreate(&ctx->ev[i]);
    for (int i = 0; i < SKR_MAX_CHUNKS && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&ctx->ev_feed[i], cudaEventDisableTiming);
    for (int i = 0; i < SKR_MAX_CHUNKS && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&ctx->ev_chunk[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->st_aux, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
    ctx->host_chunks = 8;
    if (const char *hc = getenv("GBIN_HOST_CHUNKS")) ctx->host_chunks = atoi(hc);
    if (ctx->host_chunks < 1) ctx->host_chunks = 1;
    if (ctx->host_chunks > SKR_MAX_CHUNKS) ctx->host_chunks = SKR_MAX_CHUNKS;
    if (e == cudaSuccess) e = ctx->misc.ensure(sizeof(Misc));
    if (e == cudaSuccess) e = ctx->h_misc.ensure(sizeof(Misc) + sizeof(XchgResult));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        delete ctx;
        return GBIN_E_CUDA;
    }
    *out = ctx;
    return GBIN_OK;
}

void gbin_destroy(gbin_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    cudaStreamSynchronize(ctx->stream);
    gbin_xchg_destroy(ctx);
    ctx->prof.destroy();
    for (int i = 0; i < EV_COUNT; i++) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < SKR_MAX_CHUNKS; i++) {
        cudaEventDestroy(ctx->ev_feed[i]);
        cudaEventDestroy(ctx->ev_chunk[i]);
    }
    cudaEventDestroy(ctx->ev_copy);
    cudaEventDestroy(ctx->ev_fork);
    cudaEventDestroy(ctx->ev_join);
    cudaStreamDestroy(ctx->st_aux);
    cudaStreamDestroy(ctx->st_h2d);
    cudaStreamDestroy(ctx->st_d2h);
    cudaStreamDestroy(ctx->stream);
    delete ctx;  // the buffers free their memory
}

int gbin_get_config(const gbin_ctx *ctx, gbin_config *out) {
    if (!ctx || !out) return GBIN_E_INVALID_ARG;
    *out = ctx->cfg;
    return GBIN_OK;
}

int gbin_get_timings(const gbin_ctx *ctx, gbin_timings *out) {
    if (!ctx || !out) return GBIN_E_INVALID_ARG;
    *out = ctx->tm;
    return GBIN_OK;
}

uint32_t gbin_max_read_len(void) {
    const uint32_t hw = scan_reads_max_len();  // what one warp's shared memory holds in the instance-record scan
    return hw < (uint32_t)GBIN_MAX_READ_LEN ? hw : (uint32_t)GBIN_MAX_READ_LEN;
}

uint32_t gbin_record_bytes(const gbin_ctx *ctx) { return ctx ? (uint32_t)(8 * ctx->KW + 8) : 0; }

void *gbin_pinned_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return p;
}
void gbin_pinned_free(void *p) {
    if (p) cudaFreeHost(p);
}

static void finish_timings(gbin_ctx *ctx, int launches, bool host_path) {
    auto ms = [&](int a, int b) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, ctx->ev[a], ctx->ev[b]) != cudaSuccess) {
            (void)cudaGetLastError();
            t = 0.f;
        }
        return t;
    };
    ctx->tm.h2d_ms = host_path ? ms(EV_START, EV_READS_ON_DEVICE) : 0.f;
    ctx->tm.scan_ms = ms(EV_READS_ON_DEVICE, EV_SCANNED);
    ctx->tm.sort_ms = ms(EV_SCANNED, EV_SORTED);
    ctx->tm.group_ms = ms(EV_SORTED, EV_GROUPED);
    ctx->tm.d2h_ms = host_path ? ms(EV_GROUPED, EV_TABLE_ON_HOST) : 0.f;
    ctx->tm.total_ms = ms(EV_START, host_path ? EV_TABLE_ON_HOST : EV_GROUPED);
    ctx->tm.kernel_launches = (uint32_t)launches;
    ctx->prof.collect();
}

int gbin_get_run_stats(const gbin_ctx *ctx, gbin_run_stats *out) {
    if (!ctx || !out) return GBIN_E_INVALID_ARG;
    *out = ctx->rs;
    return GBIN_OK;
}

int gbin_set_pipeline(gbin_ctx *ctx, int pipeline) {
    if (!ctx || pipeline < 1 || pipeline > 3) return GBIN_E_INVALID_ARG;
    ctx->pipeline = pipeline;
    return GBIN_OK;
}

int gbin_donate_scratch(gbin_ctx *ctx, void *d_ptr, uint64_t bytes) {
    if (!ctx) return GBIN_E_INVALID_ARG;
    ctx->donated = bytes ? d_ptr : nullptr;
    ctx->donated_bytes = d_ptr ? bytes : 0;
    return GBIN_OK;
}

int gbin_set_tuning(gbin_ctx *ctx, const char *name, int value) {
    if (!ctx || !name) return GBIN_E_INVALID_ARG;
    if (!strcmp(name, "v3_cap")) {
        if (value != 0 && value != 512 && value != 1024) return GBIN_E_INVALID_ARG;
        ctx->v3_cap = value;
    } else if (!strcmp(name, "v3_nc")) {
        if (value != 0 && value != 1 && value != 2) return GBIN_E_INVALID_ARG;
        ctx->v3_nc = value;
        ctx->v3_auto_n = 0;
    } else if (!strcmp(name, "v3_h")) {
        if (value < 0 || value > 15) return GBIN_E_INVALID_ARG;
        ctx->v3_h = value;
    } else if (!strcmp(name, "v3_pass_max")) {
        if (value < 1000) return GBIN_E_INVALID_ARG;
        ctx->v3_pass_max = (uint64_t)value;
    } else if (!strcmp(name, "xchg_timeout_ms")) {  // how long the exchange kernels wait for a peer's flag before they give up (status 2)
        if (value < 100) return GBIN_E_INVALID_ARG;
        ctx->xchg_timeout_ms = value;
        ctx->xg.plan.timeout_cycles = (long long)value * 2000000ll;
    } else if (!strcmp(name, "host_chunks")) {
        if (value < 1 || value > SKR_MAX_CHUNKS) return GBIN_E_INVALID_ARG;
        ctx->host_chunks = value;
    } else {
        return GBIN_E_INVALID_ARG;
    }
    return GBIN_OK;
}

int gbin_get_pipeline_info(const gbin_ctx *ctx, int *configured, int *last_used, uint32_t *fallbacks) {
    if (!ctx) return GBIN_E_INVALID_ARG;
    if (configured) *configured = ctx->pipeline;
    if (last_used) *last_used = ctx->last_pipeline;
    if (fallbacks) *fallbacks = ctx->fallbacks;
    return GBIN_OK;
}

int gbin_set_kernel_profiling(gbin_ctx *ctx, int enable) {
    if (!ctx) return GBIN_E_INVALID_ARG;
    ctx->prof.enabled = enable != 0;
    ctx->prof.reset();
    return GBIN_OK;
}

int gbin_get_kernel_profile(const gbin_ctx *ctx, gbin_kernel_profile *out) {
    if (!ctx || !out) return GBIN_E_INVALID_ARG;
    for (int i = 0; i < GBIN_KERNEL_KINDS; i++) {
        out->ms[i] = i < KK_COUNT ? ctx->prof.ms[i] : 0.f;
        out->launches[i] = i < KK_COUNT ? ctx->prof.launches[i] : 0u;
    }
    return GBIN_OK;
}

const char *gbin_kernel_kind_name(int kind) {
    static const char *names[] = {"scan_reads", "radix_hist", "radix_tile_scan", "radix_scatter", "find_runs", "prune_offsets", "emit_table",
                                  "skr_scan", "skr_plan", "skr_group", "v3_entries", "v3_span"};
    return (kind >= 0 && kind < KK_COUNT) ? names[kind] : "";
}

int gbin_bin_reads_device(gbin_ctx *ctx, const gbin_reads *reads, void *stream, gbin_table *out) {
    if (!ctx || !reads || !out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int launches = 0;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    int rc = bin_device_impl(ctx, reads, st, out, &launches);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    finish_timings(ctx, launches, false);
    return GBIN_OK;
}

// Copies what the sink has not streamed yet of the device table `dev` into the context's pinned arenas (regrown when too
// small — then everything is copied) plus the bucket directory, and fills *out.  Work is enqueued on st; the caller syncs.
static int table_to_pinned(gbin_ctx *ctx, const gbin_table &dev, HostSink *sink, cudaStream_t st, gbin_table *out) {
    const uint64_t B = dev.n_buckets, S = dev.n_kmers, NS = dev.n_ids;
    const int KW = dev.kmer_words;
    uint64_t s0 = sink ? sink->kmers_done : 0, n0 = sink ? sink->ids_done : 0;
    if (s0 > S || n0 > NS) s0 = n0 = 0;
    if (s0 || n0) {  // the streamed copies must have landed before the arena is handed out
        CU(cudaEventRecord(ctx->ev_copy, ctx->st_d2h));
        CU(cudaStreamWaitEvent(st, ctx->ev_copy, 0));
    }
    const size_t need_kc = (S * KW + 1) * sizeof(uint64_t), need_ko = (S + 1) * sizeof(uint64_t), need_id = (NS + 1) * sizeof(int32_t);
    if (need_kc > ctx->h_kmer_codes.cap || need_ko > ctx->h_kmer_id_off.cap || need_id > ctx->h_read_ids.cap) {
        CU(cudaStreamSynchronize(ctx->st_d2h));  // regrowing frees the arenas: nothing may be in flight into them
        CU(ctx->h_kmer_codes.ensure(need_kc));
        CU(ctx->h_kmer_id_off.ensure(need_ko));
        CU(ctx->h_read_ids.ensure(need_id));
        s0 = n0 = 0;
    }
    const size_t sz_mo = (B + 1) * sizeof(uint64_t);
    CU(ctx->h_result.ensure(sz_mo + (B + 1) * sizeof(uint32_t) + 64));
    *out = dev;
    out->on_device = 0;
    out->ctx_owned = 1;
    out->kmer_codes = static_cast<uint64_t *>(ctx->h_kmer_codes.p);
    out->kmer_id_off = static_cast<uint64_t *>(ctx->h_kmer_id_off.p);
    out->read_ids = static_cast<int32_t *>(ctx->h_read_ids.p);
    out->mmer_kmer_off = static_cast<uint64_t *>(ctx->h_result.p);
    out->mmer_codes = reinterpret_cast<uint32_t *>(static_cast<char *>(ctx->h_result.p) + sz_mo);
    if (S > s0) CU(cudaMemcpyAsync(out->kmer_codes + s0 * KW, dev.kmer_codes + s0 * KW, (S - s0) * KW * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out->kmer_id_off + s0, dev.kmer_id_off + s0, (S + 1 - s0) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (NS > n0) CU(cudaMemcpyAsync(out->read_ids + n0, dev.read_ids + n0, (NS - n0) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out->mmer_kmer_off, dev.mmer_kmer_off, (B + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (B) CU(cudaMemcpyAsync(out->mmer_codes, dev.mmer_codes, B * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return GBIN_OK;
}

int gbin_bin_reads_host(gbin_ctx *ctx, const gbin_reads *reads, gbin_table *out) {
    if (!ctx || !reads || !out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, nullptr, &st));
    int launches = 0;
    gbin_reads d = *reads;
    HostFeed feed{};
    bool use_feed = false;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    if (reads->n_reads) {
        if (!reads->data || reads->data_bytes == 0) return fail(ctx, GBIN_E_INVALID_ARG, "host reads need data and data_bytes");
        CU(ctx->d_reads.ensure(reads->data_bytes + 64));
        d.data = ctx->d_reads.as<char>();
        if (!reads->starts && reads->stride >= reads->read_len && (reads->n_reads - 1) * reads->stride + reads->read_len <= reads->data_bytes) {
            // fixed stride: read ranges are byte ranges, so the copy is left to the scan stage, which overlaps it with the scan
            feed = HostFeed{reads->data, ctx->d_reads.as<char>(), reads->data_bytes, ctx->host_chunks};
            if (reads->n_reads < 4096u * (uint64_t)feed.chunks) feed.chunks = 1;
            use_feed = true;
            CU(cudaStreamWaitEvent(ctx->st_h2d, ctx->ev[EV_START], 0));
        } else {
            CU(cudaMemcpyAsync(ctx->d_reads.p, reads->data, reads->data_bytes, cudaMemcpyHostToDevice, st));
        }
        if (reads->starts) {
            if (!reads->lens) return fail(ctx, GBIN_E_INVALID_ARG, "ragged reads need lens");
            CU(ctx->d_starts.ensure(reads->n_reads * sizeof(uint64_t)));
            CU(ctx->d_lens.ensure(reads->n_reads * sizeof(uint32_t)));
            CU(cudaMemcpyAsync(ctx->d_starts.p, reads->starts, reads->n_reads * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(ctx->d_lens.p, reads->lens, reads->n_reads * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            d.starts = ctx->d_starts.as<uint64_t>();
            d.lens = ctx->d_lens.as<uint32_t>();
            if (d.max_read_len == 0) {  // known on the host: spare the device reduction
                uint32_t mx = 0;
                for (uint64_t i = 0; i < reads->n_reads; i++) {
                    if (reads->lens[i] > mx) mx = reads->lens[i];
                    if (reads->data_bytes && reads->starts[i] + reads->lens[i] > reads->data_bytes)
                        return fail(ctx, GBIN_E_INVALID_ARG, "read %llu exceeds data_bytes", (unsigned long long)i);
                }
                d.max_read_len = mx ? mx : 1;
            }
        }
        if (reads->read_ids) {
            CU(ctx->d_ids.ensure(reads->n_reads * sizeof(int32_t)));
            CU(cudaMemcpyAsync(ctx->d_ids.p, reads->read_ids, reads->n_reads * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            d.read_ids = ctx->d_ids.as<int32_t>();
        }
    }
    if (!use_feed) CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    // the big arrays of the table are streamed into the pinned arenas as far as these reach (they are sized by the previous
    // call, so the first call on a context copies everything at the end and later calls of similar size overlap the copy)
    HostSink sink{static_cast<uint64_t *>(ctx->h_kmer_codes.p), static_cast<uint64_t *>(ctx->h_kmer_id_off.p), static_cast<int32_t *>(ctx->h_read_ids.p),
                  0, 0, 0, 0, ctx->host_chunks};
    sink.kmer_cap = ctx->h_kmer_codes.cap / (sizeof(uint64_t) * ctx->KW);
    if (ctx->h_kmer_id_off.cap / sizeof(uint64_t) < sink.kmer_cap) sink.kmer_cap = ctx->h_kmer_id_off.cap / sizeof(uint64_t);
    sink.id_cap = ctx->h_read_ids.cap / sizeof(int32_t);
    gbin_table dev;
    int rc = bin_device_impl(ctx, &d, st, &dev, &launches, use_feed ? &feed : nullptr, &sink);
    if (rc) {
        cudaStreamSynchronize(ctx->st_h2d);
        cudaStreamSynchronize(ctx->st_d2h);
        return rc;
    }
    rc = table_to_pinned(ctx, dev, &sink, st, out);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_TABLE_ON_HOST], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaStreamSynchronize(ctx->st_d2h));
    finish_timings(ctx, launches, true);
    return GBIN_OK;
}

int gbin_table_to_pinned(gbin_ctx *ctx, const gbin_table *dev, void *stream, gbin_table *host) {
    if (!ctx || !dev || !host || !dev->on_device) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int rc = table_to_pinned(ctx, *dev, nullptr, st, host);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    return GBIN_OK;
}


// ---------------------------------------------------------------- main's read loop on the device (SURVEY 8 f2)

namespace {
// d_data: the file image in device memory.  Fills *out with the ragged-reads form (device pointers owned by the context).
int split_reads_impl(gbin_ctx *ctx, const char *d_data, uint64_t size, int read_length_define, cudaStream_t st, gbin_reads *out, int *launches) {
    if (read_length_define < 2) return fail(ctx, GBIN_E_INVALID_ARG, "READ_LENGTH must be at least 2 (fgets stores READ_LENGTH-1 bytes)");
    memset(out, 0, sizeof *out);
    out->data = d_data;
    out->data_bytes = size;
    if (size == 0) return GBIN_OK;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    const uint8_t *data = reinterpret_cast<const uint8_t *>(d_data);
    const uint32_t tiles = split_tiles(size);
    const uint32_t cap = (uint32_t)read_length_define - 1u;
    CU(ctx->split_tiles_buf.ensure(((size_t)tiles + scan_scratch_elems(tiles) + 16) * sizeof(uint32_t)));
    uint32_t *tile_counts = ctx->split_tiles_buf.as<uint32_t>();
    *launches += split_find_newlines(data, size, tile_counts, tile_counts + tiles, nullptr, &dm->split_n_nl, false, st);
    CU(cudaGetLastError());
    // the last line may lack its newline: it still is a line for fgets
    CU(cudaMemcpyAsync(&hm->last_byte, d_data + size - 1, 1, cudaMemcpyDeviceToHost, st));
    CU(read_back(ctx, &Misc::split_n_nl, st));
    const uint64_t n_nl = hm->split_n_nl;
    const uint64_t n_lines = n_nl + (hm->last_byte != '\n' ? 1 : 0);
    if (n_lines >= (1ull << 32) - 1) return fail(ctx, GBIN_E_TOO_LARGE, "more than 2^32-1 lines in one file image");
    CU(ctx->split_nl.ensure((n_nl + 1) * sizeof(uint64_t)));
    *launches += split_find_newlines(data, size, tile_counts, nullptr, ctx->split_nl.as<uint64_t>(), nullptr, true, st);
    CU(ctx->split_base.ensure((n_lines + 1) * sizeof(uint32_t)));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(n_lines)));
    *launches += split_count_reads(ctx->split_nl.as<uint64_t>(), n_nl, size, cap, n_lines, ctx->split_base.as<uint32_t>(),
                                   ctx->scan_scratch.as<uint32_t>(), &dm->split_n_reads, st);
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::split_n_reads, st));
    const uint64_t n_reads = hm->split_n_reads;
    CU(ctx->d_starts.ensure((n_reads + 1) * sizeof(uint64_t)));
    CU(ctx->d_lens.ensure((n_reads + 1) * sizeof(uint32_t)));
    *launches += split_emit_reads(ctx->split_nl.as<uint64_t>(), n_nl, size, cap, n_lines, ctx->split_base.as<uint32_t>(), ctx->d_starts.as<uint64_t>(),
                                  ctx->d_lens.as<uint32_t>(), st);
    CU(cudaGetLastError());
    out->n_reads = n_reads;
    out->starts = ctx->d_starts.as<uint64_t>();
    out->lens = ctx->d_lens.as<uint32_t>();
    out->max_read_len = 0;  // the reads are at most cap - 1 bases long, usually far shorter: the binning call finds the real maximum on the device
    return GBIN_OK;
}
}  // namespace

int gbin_copy_to_host(gbin_ctx *ctx, void *host_dst, const void *device_src, uint64_t bytes) {
    if (!ctx || (bytes && (!host_dst || !device_src))) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    CU(cudaStreamSynchronize(ctx->stream));
    if (bytes) CU(cudaMemcpy(host_dst, device_src, bytes, cudaMemcpyDeviceToHost));
    return GBIN_OK;
}

int gbin_split_reads_device(gbin_ctx *ctx, const char *d_data, uint64_t data_bytes, int read_length_define, void *stream, gbin_reads *out) {
    if (!ctx || !out || (data_bytes && !d_data)) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int launches = 0;
    int rc = split_reads_impl(ctx, d_data, data_bytes, read_length_define, st, out, &launches);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    ctx->tm.kernel_launches = (uint32_t)launches;
    return GBIN_OK;
}

int gbin_bin_file_host(gbin_ctx *ctx, const char *path, int read_length_define, gbin_table *out) {
    if (!ctx || !path || !out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, nullptr, &st));
    FILE *f = fopen(path, "rb");
    if (!f) return fail(ctx, GBIN_E_IO, "cannot open %s", path);
    if (fseek(f, 0, SEEK_END) != 0) {
        fclose(f);
        return fail(ctx, GBIN_E_IO, "cannot seek in %s", path);
    }
    const long fsize = ftell(f);
    rewind(f);
    if (fsize < 0) {
        fclose(f);
        return fail(ctx, GBIN_E_IO, "cannot size %s", path);
    }
    const uint64_t size = (uint64_t)fsize;
    cudaError_t e = ctx->h_file.ensure(size + 64);
    if (e == cudaSuccess) e = ctx->d_reads.ensure(size + 64);
    if (e != cudaSuccess) {
        fclose(f);
        (void)cudaGetLastError();
        return fail(ctx, GBIN_E_NOMEM, "no room for the image of %s (%llu bytes)", path, (unsigned long long)size);
    }
    const size_t got = size ? fread(ctx->h_file.p, 1, size, f) : 0;
    fclose(f);
    if (got != size) return fail(ctx, GBIN_E_IO, "short read on %s", path);
    int launches = 0;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    if (size) CU(cudaMemcpyAsync(ctx->d_reads.p, ctx->h_file.p, size, cudaMemcpyHostToDevice, st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    gbin_reads rd;
    int rc = split_reads_impl(ctx, ctx->d_reads.as<char>(), size, read_length_define, st, &rd, &launches);
    if (rc) return rc;
    gbin_table dev;
    rc = bin_device_impl(ctx, &rd, st, &dev, &launches);
    if (rc) return rc;
    rc = table_to_pinned(ctx, dev, nullptr, st, out);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_TABLE_ON_HOST], st));
    CU(cudaStreamSynchronize(st));
    finish_timings(ctx, launches, true);
    return GBIN_OK;
}

int gbin_table_digest(gbin_ctx *ctx, const gbin_table *t, void *stream, uint64_t *digest_out) {
    if (!t || !digest_out) return GBIN_E_INVALID_ARG;
    if (!t->on_device) {
        *digest_out = table_digest_host(t);
        return GBIN_OK;
    }
    if (!ctx) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    table_digest_device(t, &ctx->misc.as<Misc>()->digest, st);
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::digest, st));
    *digest_out = static_cast<Misc *>(ctx->h_misc.p)->digest;
    return GBIN_OK;
}

int gbin_expand_read_ids_device(gbin_ctx *ctx, const gbin_table *t, void *stream, gbin_expanded *out) {
    if (!ctx || !t || !out || !t->on_device) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    const uint64_t K = (uint64_t)t->kmer_size, S = t->n_kmers, N = t->n_ids;
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t need = (S * K + 1) * sizeof(uint64_t) + (K * N + 1) * sizeof(int32_t);
    if (need > (uint64_t)free_b + ctx->x_list_off.cap + ctx->x_ids.cap)
        return fail(ctx, GBIN_E_TOO_LARGE, "expanded id lists need %llu bytes (K = %llu copies of %llu ids), %llu are free", (unsigned long long)need,
                    (unsigned long long)K, (unsigned long long)N, (unsigned long long)free_b);
    CU(ctx->x_list_off.ensure((S * K + 1) * sizeof(uint64_t)));
    CU(ctx->x_ids.ensure((K * N + 1) * sizeof(int32_t)));
    expand_ids_device(t->kmer_id_off, t->read_ids, S, (uint32_t)K, ctx->x_list_off.as<uint64_t>(), ctx->x_ids.as<int32_t>(), ctx->sm_count, st);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    out->kmer_size = t->kmer_size;
    out->on_device = 1;
    out->n_lists = S * K;
    out->n_ids = K * N;
    out->list_off = ctx->x_list_off.as<uint64_t>();
    out->ids = ctx->x_ids.as<int32_t>();
    return GBIN_OK;
}

int gbin_expanded_to_host(gbin_ctx *ctx, const gbin_expanded *dev, gbin_expanded *host) {
    if (!ctx || !dev || !host || !dev->on_device) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    *host = *dev;
    host->on_device = 0;
    host->list_off = static_cast<uint64_t *>(malloc((dev->n_lists + 1) * sizeof(uint64_t)));
    host->ids = static_cast<int32_t *>(malloc((dev->n_ids + 1) * sizeof(int32_t)));
    if (!host->list_off || !host->ids) {
        free(host->list_off);
        free(host->ids);
        host->list_off = nullptr;
        host->ids = nullptr;
        return GBIN_E_NOMEM;
    }
    CU(cudaMemcpy(host->list_off, dev->list_off, (dev->n_lists + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (dev->n_ids) CU(cudaMemcpy(host->ids, dev->ids, dev->n_ids * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return GBIN_OK;
}

int gbin_table_to_host(gbin_ctx *ctx, const gbin_table *dev, gbin_table *host) {
    if (!ctx || !dev || !host || !dev->on_device) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    const uint64_t B = dev->n_buckets, S = dev->n_kmers, NS = dev->n_ids;
    const int KW = dev->kmer_words;
    *host = *dev;
    host->on_device = 0;
    host->ctx_owned = 0;
    host->mmer_codes = static_cast<uint32_t *>(malloc((B + 1) * sizeof(uint32_t)));
    host->mmer_kmer_off = static_cast<uint64_t *>(malloc((B + 1) * sizeof(uint64_t)));
    host->kmer_codes = static_cast<uint64_t *>(malloc((S * KW + 1) * sizeof(uint64_t)));
    host->kmer_id_off = static_cast<uint64_t *>(malloc((S + 1) * sizeof(uint64_t)));
    host->read_ids = static_cast<int32_t *>(malloc((NS + 1) * sizeof(int32_t)));
    if (!host->mmer_codes || !host->mmer_kmer_off || !host->kmer_codes || !host->kmer_id_off || !host->read_ids) {
        gbin_table_free(host);
        return fail(ctx, GBIN_E_NOMEM, "host table allocation failed");
    }
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaMemcpy(host->mmer_codes, dev->mmer_codes, B * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host->mmer_kmer_off, dev->mmer_kmer_off, (B + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host->kmer_codes, dev->kmer_codes, S * KW * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host->kmer_id_off, dev->kmer_id_off, (S + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(host->read_ids, dev->read_ids, NS * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return GBIN_OK;
}

// ---------------------------------------------------------------- staged entry points (multi-GPU path)

int gbin_count_instances_device(gbin_ctx *ctx, const gbin_reads *reads, void *stream, uint64_t *n_out) {
    if (!ctx || !reads || !n_out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint32_t max_len = 0;
    int launches = 0;
    return plan_reads(ctx, reads, st, n_out, &max_len, &launches);
}

int gbin_scan_reads_device(gbin_ctx *ctx, const gbin_reads *reads, uint32_t arrival_base, void *d_records, uint64_t capacity,
                           void *stream, uint64_t *n_out) {
    if (!ctx || !reads || !n_out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint64_t n = 0;
    uint32_t max_len = 0;
    int launches = 0;
    int rc = plan_reads(ctx, reads, st, &n, &max_len, &launches);
    if (rc) return rc;
    if (max_len > GBIN_MAX_READ_LEN) return fail(ctx, GBIN_E_TOO_LARGE, "read length %u exceeds GBIN_MAX_READ_LEN", max_len);
    if (n > capacity) return fail(ctx, GBIN_E_INVALID_ARG, "record buffer too small: need %llu", (unsigned long long)n);
    if (n && !d_records) return GBIN_E_INVALID_ARG;
    rc = run_scan(ctx, reads, arrival_base, d_records, max_len, st, &launches);
    if (rc) return rc;
    CU(read_back(ctx, &Misc::grp, st));
    ctx->prof.collect();
    const unsigned long long bad = static_cast<Misc *>(ctx->h_misc.p)->grp.bad_bases;
    if (bad) return fail(ctx, GBIN_E_NON_ACGT, "%llu bases other than A/C/G/T in the batch", bad);
    *n_out = n;
    ctx->tm.kernel_launches = (uint32_t)launches;
    return GBIN_OK;
}

int gbin_partition_records_device(gbin_ctx *ctx, const void *d_records, uint64_t n, uint32_t n_parts, void *d_out, void *stream,
                                  uint64_t *counts_host) {
    return partition_by_owner(ctx, n, n_parts, stream, counts_host, [&](void *scratch, uint64_t *d_counts, cudaStream_t st) {
        return radix_partition_by_owner(d_records, d_out, n, ctx->KW, n_parts, scratch, d_counts, st);
    });
}

// ---------------------------------------------------------------- owner exchange over peer memory

namespace {
struct XchgHandle {  // what a rank publishes: GBIN_XCHG_HANDLE_BYTES
    cudaIpcMemHandle_t recv, shared;
    uint64_t cap;
    uint32_t rank, world;
    uint32_t record_bytes, magic;
};
static_assert(sizeof(XchgHandle) <= GBIN_XCHG_HANDLE_BYTES, "handle blob size");
constexpr uint32_t XCHG_MAGIC = 0x67786331u;

// Starts the context's exchange plan over its own buffers; the caller fills in the peers' (cap, peer_recv, peer_sh).
void init_xchg_plan(gbin_ctx *ctx) {
    auto &x = ctx->xg;
    if (x.n_opened) gbin_xchg_detach(ctx);  // a second attach replaces the first one's mappings
    memset(&x.plan, 0, sizeof x.plan);
    x.plan.timeout_cycles = (long long)ctx->xchg_timeout_ms * 2000000ll;  // about 2 GHz
    x.plan.rank = x.rank;
    x.plan.world = x.world;
    x.plan.dst_tab = x.dst_tab;
    x.plan.result = x.result;
}
}  // namespace

int gbin_xchg_create(gbin_ctx *ctx, uint32_t rank, uint32_t world, uint64_t capacity_records, void *handle_out) {
    if (!ctx || !handle_out || world == 0 || world > (uint32_t)XCHG_MAX_WORLD || rank >= world || capacity_records == 0) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    gbin_xchg_destroy(ctx);
    auto &x = ctx->xg;
    const size_t rb = gbin_skr_record_bytes(ctx);
    CU(cudaMalloc(&x.recv, (capacity_records + 1) * rb));
    CU(cudaMalloc(reinterpret_cast<void **>(&x.sh), sizeof(XchgShared)));
    CU(cudaMalloc(reinterpret_cast<void **>(&x.dst_tab), sizeof(char *) * XCHG_MAX_WORLD));
    CU(cudaMalloc(reinterpret_cast<void **>(&x.result), sizeof(XchgResult)));
    CU(cudaMemset(x.sh, 0, sizeof(XchgShared)));
    CU(cudaMemset(x.result, 0, sizeof(XchgResult)));
    x.rank = rank;
    x.world = world;
    x.cap = capacity_records;
    x.epoch = 0;
    x.created = true;
    XchgHandle h;
    memset(&h, 0, sizeof h);
    CU(cudaIpcGetMemHandle(&h.recv, x.recv));
    CU(cudaIpcGetMemHandle(&h.shared, x.sh));
    h.cap = capacity_records;
    h.rank = rank;
    h.world = world;
    h.record_bytes = (uint32_t)rb;
    h.magic = XCHG_MAGIC;
    memset(handle_out, 0, GBIN_XCHG_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof h);
    return GBIN_OK;
}

int gbin_xchg_attach(gbin_ctx *ctx, const void *all_handles) {
    if (!ctx || !all_handles || !ctx->xg.created) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    auto &x = ctx->xg;
    init_xchg_plan(ctx);
    for (uint32_t r = 0; r < x.world; r++) {
        XchgHandle h;
        memcpy(&h, static_cast<const char *>(all_handles) + (size_t)r * GBIN_XCHG_HANDLE_BYTES, sizeof h);
        if (h.magic != XCHG_MAGIC || h.rank != r || h.world != x.world || h.record_bytes != gbin_skr_record_bytes(ctx))
            return fail(ctx, GBIN_E_INVALID_ARG, "exchange handle %u does not match this context (rank/world/record size)", r);
        x.plan.cap[r] = h.cap;
        if (r == x.rank) {
            x.plan.peer_recv[r] = x.recv;
            x.plan.peer_sh[r] = x.sh;
            continue;
        }
        void *pr = nullptr, *ps = nullptr;
        CU(cudaIpcOpenMemHandle(&pr, h.recv, cudaIpcMemLazyEnablePeerAccess));
        x.opened[x.n_opened++] = pr;
        CU(cudaIpcOpenMemHandle(&ps, h.shared, cudaIpcMemLazyEnablePeerAccess));
        x.opened[x.n_opened++] = ps;
        x.plan.peer_recv[r] = pr;
        x.plan.peer_sh[r] = static_cast<XchgShared *>(ps);
    }
    x.attached = true;
    return GBIN_OK;
}

// Phase 1 of a collective teardown: close the mappings of the peers' buffers.  Every rank detaches, the caller barriers, and only then
// does an owner free what it exported (gbin_xchg_destroy): freeing exported memory while an importer still has it open is undefined.
void gbin_xchg_detach(gbin_ctx *ctx) {
    if (!ctx || !ctx->xg.created) return;
    auto &x = ctx->xg;
    cudaSetDevice(ctx->cfg.device);
    cudaDeviceSynchronize();
    for (int i = 0; i < x.n_opened; i++) cudaIpcCloseMemHandle(x.opened[i]);
    x.n_opened = 0;
    x.attached = false;
    (void)cudaGetLastError();
}

void gbin_xchg_destroy(gbin_ctx *ctx) {
    if (!ctx || !ctx->xg.created) return;
    auto &x = ctx->xg;
    gbin_xchg_detach(ctx);
    cudaFree(x.recv);
    cudaFree(x.sh);
    cudaFree(x.dst_tab);
    cudaFree(x.result);
    x.recv = nullptr;
    x.sh = nullptr;
    x.dst_tab = nullptr;
    x.result = nullptr;
    x.created = x.attached = false;
    (void)cudaGetLastError();
}

int gbin_xchg_exchange_skr(gbin_ctx *ctx, const void *d_skr, uint64_t n, void *stream, void **d_recv_out, uint64_t *n_recv_out,
                           uint64_t *sent_counts) {
    if (!ctx || !d_recv_out || !n_recv_out || (n && !d_skr)) return GBIN_E_INVALID_ARG;
    if (!ctx->xg.attached) return fail(ctx, GBIN_E_STATE, "gbin_xchg_exchange_skr before gbin_xchg_create / gbin_xchg_attach");
    if (n >= (1ull << 32) - 8192) return fail(ctx, GBIN_E_TOO_LARGE, "too many records in one exchange call");
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    auto &x = ctx->xg;
    CU(ctx->radix_scratch.ensure(radix_scratch_bytes(n)));
    x.plan.epoch = ++x.epoch;
    const int launches = radix_exchange_skr_by_owner(d_skr, n, ctx->cfg.kmer_size <= 32 ? 8 : 12, ctx->radix_scratch.p, x.plan, st);
    CU(cudaGetLastError());
    XchgResult *hr = reinterpret_cast<XchgResult *>(static_cast<char *>(ctx->h_misc.p) + sizeof(Misc));
    CU(cudaMemcpyAsync(hr, x.result, sizeof(XchgResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->tm.kernel_launches = (uint32_t)launches;
    if (sent_counts)
        for (uint32_t r = 0; r < x.world; r++) sent_counts[r] = hr->sent[r];
    if (hr->status == 2u) return fail(ctx, GBIN_E_CUDA, "owner exchange: a peer did not answer within the time limit");
    if (hr->status == 1u) return fail(ctx, GBIN_E_TOO_LARGE, "owner exchange: a receive buffer is too small for this batch");
    *d_recv_out = x.recv;
    *n_recv_out = hr->n_in;
    return GBIN_OK;
}

uint32_t gbin_owner_of(uint32_t mmer_code, uint32_t n_parts) { return n_parts ? owner_of_mmer(mmer_code, n_parts) : 0u; }

uint32_t gbin_skr_record_bytes(const gbin_ctx *ctx) { return ctx ? (ctx->cfg.kmer_size <= 32 ? 32u : 48u) : 0u; }

int gbin_scan_skr_device(gbin_ctx *ctx, const gbin_reads *reads, uint32_t arrival_base, void *d_skr, uint64_t capacity, void *stream,
                         uint64_t *n_skr_out, uint64_t *n_instances_out) {
    if (!ctx || !reads || !n_skr_out) return GBIN_E_INVALID_ARG;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint64_t n = 0, n_skr = 0;
    uint32_t max_len = 0;
    int launches = 0;
    int rc = plan_reads(ctx, reads, st, &n, &max_len, &launches);
    if (rc) return rc;
    if (max_len > GBIN_MAX_READ_LEN) return fail(ctx, GBIN_E_TOO_LARGE, "read length %u exceeds GBIN_MAX_READ_LEN", max_len);
    if (n && !d_skr) return GBIN_E_INVALID_ARG;
    if (n) {
        rc = run_skr_scan(ctx, reads, n, max_len, arrival_base, d_skr, capacity, st, &n_skr, &launches);
        if (rc) return rc;
    }
    ctx->prof.collect();
    *n_skr_out = n_skr;
    if (n_instances_out) *n_instances_out = n;
    ctx->tm.kernel_launches = (uint32_t)launches;
    return GBIN_OK;
}

int gbin_partition_skr_device(gbin_ctx *ctx, const void *d_skr, uint64_t n, uint32_t n_parts, void *d_out, void *stream, uint64_t *counts_host) {
    return partition_by_owner(ctx, n, n_parts, stream, counts_host, [&](void *scratch, uint64_t *d_counts, cudaStream_t st) {
        return radix_partition_skr_by_owner(d_skr, d_out, n, ctx->cfg.kmer_size <= 32 ? 8 : 12, n_parts, scratch, d_counts, st);
    });
}

int gbin_group_skr_device(gbin_ctx *ctx, void *d_skr, uint64_t n_skr, const int32_t *d_ids_by_arrival, int32_t id_base, void *stream,
                          gbin_table *out, int *used_fallback) {
    if (!ctx || !out || (n_skr && !d_skr)) return GBIN_E_INVALID_ARG;
    if (n_skr >= (1ull << 31)) return fail(ctx, GBIN_E_TOO_LARGE, "too many super-k-mer records in one call");
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int launches = 0;
    if (used_fallback) *used_fallback = 0;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    CU(cudaEventRecord(ctx->ev[EV_SCANNED], st));
    bool done = false;
    uint64_t n = 0;
    int used = 2;
    if (n_skr) {
        int rc = run_skr_group(ctx, d_skr, n_skr, d_ids_by_arrival, id_base, st, out, &launches, &done, &n, nullptr, &used);
        if (rc) return rc;
        if (!done) {
            // A unit overflowed (one k-mer with more instances than a unit holds).  The records were consumed by the sort,
            // so the caller re-runs the batch from the reads through the instance-record entry points (pipeline 1).
            if (used_fallback) *used_fallback = 1;
            return fail(ctx, GBIN_E_STATE, "a shared-memory unit overflowed; re-run this batch through gbin_group_records_device");
        }
    } else {
        CU(cudaMemsetAsync(&ctx->misc.as<Misc>()->grp.bad_bases, 0, sizeof(unsigned long long), st));
        int rc = run_group(ctx, nullptr, nullptr, 0, d_ids_by_arrival, id_base, st, out, &launches, ctx->ev[EV_SORTED]);
        if (rc) return rc;
    }
    CU(cudaEventRecord(ctx->ev[EV_GROUPED], st));
    CU(cudaStreamSynchronize(st));
    finish_timings(ctx, launches, false);
    ctx->last_pipeline = used;
    return GBIN_OK;
}

int gbin_group_records_device(gbin_ctx *ctx, void *d_records, uint64_t n, const int32_t *d_ids_by_arrival, int32_t id_base,
                              void *stream, gbin_table *out) {
    if (!ctx || !out || (n && !d_records)) return GBIN_E_INVALID_ARG;
    if (n >= (1ull << 32) - 8192) return fail(ctx, GBIN_E_TOO_LARGE, "%llu records in one group call (limit 2^32)", (unsigned long long)n);
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    const size_t rb = sizeof(uint64_t) * ctx->KW + 8;
    CU(ctx->rec_b.ensure((n + 1) * rb));
    int launches = 0;
    CU(cudaMemsetAsync(&ctx->misc.as<Misc>()->grp.bad_bases, 0, sizeof(unsigned long long), st));
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    CU(cudaEventRecord(ctx->ev[EV_SCANNED], st));
    int rc = run_group(ctx, d_records, ctx->rec_b.p, n, d_ids_by_arrival, id_base, st, out, &launches, ctx->ev[EV_SORTED]);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_GROUPED], st));
    CU(cudaStreamSynchronize(st));
    finish_timings(ctx, launches, false);
    return GBIN_OK;
}


// ---------------------------------------------------------------- several GPUs behind one C call (one process, one host thread per GPU)

struct gbin_multi {
    int n = 0;
    std::vector<gbin_ctx *> ctx;
    std::vector<int> dev;
    uint64_t xchg_cap = 0;
    char err[512] = {0};
    // A reusable barrier for the worker threads of one call.  It returns the OR of the flags all threads passed in, so that every
    // thread takes the same decision after it, even while another thread already records its status of the next step.
    std::mutex mu;
    std::condition_variable cv;
    int waiting = 0, generation = 0, flags_in = 0, flags_out = 0;
    int barrier(int flags = 0) {
        std::unique_lock<std::mutex> lk(mu);
        const int gen = generation;
        flags_in |= flags;
        if (++waiting == n) {
            flags_out = flags_in;
            flags_in = 0;
            waiting = 0;
            generation++;
            cv.notify_all();
        } else {
            cv.wait(lk, [&] { return gen != generation; });
        }
        return flags_out;  // the next generation cannot complete before this thread has arrived at it
    }
};

namespace {
// Every context's exchange plan gets the peers' buffers by address: one process, peer access enabled, no IPC handles.
int multi_attach_local(gbin_multi *m, int g) {
    gbin_ctx *ctx = m->ctx[g];
    auto &x = ctx->xg;
    init_xchg_plan(ctx);
    for (int r = 0; r < m->n; r++) {
        x.plan.cap[r] = m->ctx[r]->xg.cap;
        x.plan.peer_recv[r] = m->ctx[r]->xg.recv;
        x.plan.peer_sh[r] = m->ctx[r]->xg.sh;
    }
    x.attached = true;
    return GBIN_OK;
}
}  // namespace

int gbin_multi_create(const gbin_config *cfg, const int *devices, int n_devices, gbin_multi **out) {
    if (!cfg || !out || n_devices < 1 || n_devices > XCHG_MAX_WORLD) return GBIN_E_INVALID_ARG;
    *out = nullptr;
    gbin_multi *m = new (std::nothrow) gbin_multi();
    if (!m) return GBIN_E_NOMEM;
    m->n = n_devices;
    for (int g = 0; g < n_devices; g++) {
        gbin_config c = *cfg;
        c.device = devices ? devices[g] : g;
        gbin_ctx *ctx = nullptr;
        const int rc = gbin_create(&c, &ctx);
        if (rc) {
            gbin_multi_destroy(m);
            return rc;
        }
        m->ctx.push_back(ctx);
        m->dev.push_back(c.device);
    }
    for (int a = 0; a < n_devices; a++) {  // peer access both ways between every pair (the exchange stores into the owners' buffers)
        cudaSetDevice(m->dev[a]);
        for (int b = 0; b < n_devices; b++) {
            if (a == b) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, m->dev[a], m->dev[b]);
            if (!can) {
                gbin_multi_destroy(m);
                return GBIN_E_CUDA;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(m->dev[b], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                (void)cudaGetLastError();
                gbin_multi_destroy(m);
                return GBIN_E_CUDA;
            }
            (void)cudaGetLastError();
        }
    }
    *out = m;
    return GBIN_OK;
}

void gbin_multi_destroy(gbin_multi *m) {
    if (!m) return;
    for (gbin_ctx *c : m->ctx) {  // nobody stores into a peer's buffer any more: first let every device finish, then free
        cudaSetDevice(c->cfg.device);
        cudaDeviceSynchronize();
    }
    for (gbin_ctx *c : m->ctx) gbin_destroy(c);
    delete m;
}

const char *gbin_multi_last_error(const gbin_multi *m) { return m ? m->err : ""; }
int gbin_multi_devices(const gbin_multi *m) { return m ? m->n : 0; }
gbin_ctx *gbin_multi_context(gbin_multi *m, int i) { return (m && i >= 0 && i < m->n) ? m->ctx[i] : nullptr; }

// reads: HOST memory (pinned for the full PCIe rate).  GPU g takes the contiguous read range [g*n/G, (g+1)*n/G), runs the scan,
// sends every record to the owner of its m-mer bucket (peer stores over NVLink), groups what it received.  tables_out[g] is GPU
// g's part of the table (its own m-mer buckets) in that context's pinned arena (ctx-owned, valid until the next call).
int gbin_multi_bin_reads_host(gbin_multi *m, const gbin_reads *reads, gbin_table *tables_out) {
    if (!m || !reads || !tables_out) return GBIN_E_INVALID_ARG;
    const int G = m->n;
    const uint64_t n = reads->n_reads;
    if (n && !reads->data) return GBIN_E_INVALID_ARG;
    if (reads->starts && !reads->lens) return GBIN_E_INVALID_ARG;
    std::vector<int> rcs(G, GBIN_OK);
    std::vector<uint64_t> n_skr(G, 0);
    std::vector<uint64_t> part_counts((size_t)G * G, 0);  // [g * G + o]: instance records GPU g holds for owner o (overflow redo)
    std::vector<std::string> errs(G);
    m->err[0] = 0;
    auto work = [&](int g) {
        gbin_ctx *ctx = m->ctx[g];
        int &rc = rcs[g];
        auto failed = [&](int code, const char *what) {
            rc = code;
            errs[g] = std::string(what) + ": " + gbin_last_error(ctx);
        };
        cudaSetDevice(ctx->cfg.device);
        cudaStream_t st = ctx->stream;
        const uint64_t lo = n * g / G, hi = n * (g + 1) / G, cnt = hi - lo;
        // ---- this GPU's shard to the device
        gbin_reads d = *reads;
        d.n_reads = cnt;
        d.read_ids = nullptr;
        cudaError_t e = cudaSuccess;
        if (cnt) {
            if (!reads->starts) {
                const uint64_t b0 = lo * reads->stride, b1 = (hi - 1) * reads->stride + reads->read_len;
                e = ctx->d_reads.ensure(b1 - b0 + 64);
                if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_reads.p, reads->data + b0, b1 - b0, cudaMemcpyHostToDevice, st);
                d.data = ctx->d_reads.as<char>();
                d.data_bytes = b1 - b0;
            } else {
                uint64_t b0 = ~0ull, b1 = 0;
                for (uint64_t i = lo; i < hi; i++) {
                    if (reads->starts[i] < b0) b0 = reads->starts[i];
                    if (reads->starts[i] + reads->lens[i] > b1) b1 = reads->starts[i] + reads->lens[i];
                }
                if (b1 < b0) b0 = b1 = 0;
                std::vector<uint64_t> st_rel(cnt);
                for (uint64_t i = 0; i < cnt; i++) st_rel[i] = reads->starts[lo + i] - b0;
                e = ctx->d_reads.ensure(b1 - b0 + 64);
                if (e == cudaSuccess) e = ctx->d_starts.ensure(cnt * sizeof(uint64_t));
                if (e == cudaSuccess) e = ctx->d_lens.ensure(cnt * sizeof(uint32_t));
                if (e == cudaSuccess && b1 > b0) e = cudaMemcpyAsync(ctx->d_reads.p, reads->data + b0, b1 - b0, cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_starts.p, st_rel.data(), cnt * sizeof(uint64_t), cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_lens.p, reads->lens + lo, cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // st_rel goes out of scope
                d.data = ctx->d_reads.as<char>();
                d.data_bytes = b1 - b0;
                d.starts = ctx->d_starts.as<uint64_t>();
                d.lens = ctx->d_lens.as<uint32_t>();
                d.max_read_len = 0;
            }
        }
        const int32_t *d_ids = nullptr;
        if (e == cudaSuccess && reads->read_ids && n) {  // ids are looked up by global arrival index: every GPU holds the whole array
            e = ctx->d_ids.ensure(n * sizeof(int32_t));
            if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_ids.p, reads->read_ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, st);
            d_ids = ctx->d_ids.as<int32_t>();
        }
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            failed(e == cudaErrorMemoryAllocation ? GBIN_E_NOMEM : GBIN_E_CUDA, "copying the shard to the device");
        }
        // ---- scan into this context's record buffer (sized by an estimate, regrown to the exact need when short)
        uint64_t ninst = 0, cap = 0;
        if (!rc && cnt) {
            uint64_t est = 0;
            rc = gbin_count_instances_device(ctx, &d, st, &est);
            cap = est / 6 + cnt + 1024;
            const size_t rb = gbin_skr_record_bytes(ctx);
            for (int attempt = 0; !rc && attempt < 2; attempt++) {
                if (ctx->skr_a.ensure((cap + 1) * rb) != cudaSuccess) {
                    (void)cudaGetLastError();
                    failed(GBIN_E_NOMEM, "record buffer");
                    break;
                }
                const int r2 = gbin_scan_skr_device(ctx, &d, (uint32_t)lo, ctx->skr_a.p, cap, st, &n_skr[g], &ninst);
                if (r2 == GBIN_E_INVALID_ARG && attempt == 0 && cap < est) {
                    cap = est;  // more segments than estimated
                    continue;
                }
                if (r2) failed(r2, "scan");
                break;
            }
        } else if (!rc) {
            n_skr[g] = 0;
        }
        if (m->barrier(rc != GBIN_OK)) return;  // ---- somebody failed; else every rank knows every rank's record count
        uint64_t mx = 0;
        for (int r = 0; r < G; r++)
            if (n_skr[r] > mx) mx = n_skr[r];
        void *d_recv = nullptr;
        uint64_t n_recv = 0;
        const uint64_t want = mx + mx / 3 + 65536;
        if (G == 1) {  // nothing to exchange
            d_recv = ctx->skr_a.p;
            n_recv = n_skr[0];
        } else {
        if (!ctx->xg.created || ctx->xg.cap < want || ctx->xg.world != (uint32_t)G) {
            char blob[GBIN_XCHG_HANDLE_BYTES];
            const int r2 = gbin_xchg_create(ctx, (uint32_t)g, (uint32_t)G, want + want / 8, blob);
            if (r2) failed(r2, "exchange buffers");
        }
        if (m->barrier(rc != GBIN_OK)) return;  // ---- all buffers exist
        multi_attach_local(m, g);
        m->barrier();
        // ---- owner exchange (collective)
        const int rx = gbin_xchg_exchange_skr(ctx, ctx->skr_a.p, n_skr[g], st, &d_recv, &n_recv, nullptr);
        if (rx) failed(rx, "owner exchange");
        }
        // ---- grouping of this GPU's buckets
        gbin_table dev;
        int overflow = 0;
        if (!rc) {
            const int r2 = gbin_group_skr_device(ctx, d_recv, n_recv, d_ids, reads->id_base, st, &dev, &overflow);
            if (r2 && !(r2 == GBIN_E_STATE && overflow)) failed(r2, "grouping");
        }
        const int flags = m->barrier((rc != GBIN_OK) | (overflow ? 2 : 0));  // ---- did some rank fail, did some unit overflow
        if (flags & 1) return;
        if (flags & 2) {
            // One k-mer had more instances than a unit holds and the super-k-mer records were consumed by the sort: every GPU redoes
            // its shard in instance-record form (pipeline 1), which groups in HBM and cannot overflow.  Scan into rec_a, partition
            // into skr_a (dead now), then every owner gathers its part of every GPU's partition, in rank order, into its rec_a.
            const size_t rb = gbin_record_bytes(ctx);
            uint64_t n_rec = 0;
            if (ctx->rec_a.ensure((ninst + 1) * rb) != cudaSuccess) {
                (void)cudaGetLastError();
                failed(GBIN_E_NOMEM, "instance-record buffer");
            }
            if (!rc) {
                const int r3 = gbin_scan_reads_device(ctx, &d, (uint32_t)lo, ctx->rec_a.p, ninst, st, &n_rec);
                if (r3) failed(r3, "instance-record scan");
            }
            if (!rc && G > 1) {
                if (ctx->skr_a.ensure((n_rec + 1) * rb) != cudaSuccess) {
                    (void)cudaGetLastError();
                    failed(GBIN_E_NOMEM, "partition buffer");
                } else {
                    const int r3 = gbin_partition_records_device(ctx, ctx->rec_a.p, n_rec, (uint32_t)G, ctx->skr_a.p, st, &part_counts[(size_t)g * G]);
                    if (r3) failed(r3, "instance-record partition");
                }
            }
            if (G > 1) {
                if (m->barrier(rc != GBIN_OK)) return;  // ---- every rank's parts are in its skr_a, their sizes in part_counts
                n_rec = 0;
                for (int r = 0; r < G; r++) n_rec += part_counts[(size_t)r * G + g];
                e = ctx->rec_a.ensure((n_rec + 1) * rb);
                uint64_t at = 0;
                for (int r = 0; r < G && e == cudaSuccess; r++) {
                    uint64_t off = 0;
                    for (int o = 0; o < g; o++) off += part_counts[(size_t)r * G + o];
                    const uint64_t c = part_counts[(size_t)r * G + g];
                    if (c) e = cudaMemcpyAsync(ctx->rec_a.as<char>() + at * rb, m->ctx[r]->skr_a.as<char>() + off * rb, c * rb, cudaMemcpyDefault, st);
                    at += c;
                }
                if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // (no rank writes its skr_a again in this call)
                if (e != cudaSuccess) {
                    (void)cudaGetLastError();
                    failed(e == cudaErrorMemoryAllocation ? GBIN_E_NOMEM : GBIN_E_CUDA, "gathering the owner's records");
                }
            }
            if (rc) return;
            const int r3 = gbin_group_records_device(ctx, ctx->rec_a.p, n_rec, d_ids, reads->id_base, st, &dev);
            if (r3) {
                failed(r3, "grouping (instance records)");
                return;
            }
        }
        const int r2 = gbin_table_to_pinned(ctx, &dev, st, &tables_out[g]);
        if (r2) failed(r2, "table to host");
    };
    std::vector<std::thread> th;
    for (int g = 1; g < G; g++) th.emplace_back(work, g);
    work(0);
    for (auto &t : th) t.join();
    for (int g = 0; g < G; g++)
        if (rcs[g]) {
            snprintf(m->err, sizeof m->err, "GPU %d: %s", m->dev[g], errs[g].c_str());
            return rcs[g];
        }
    return GBIN_OK;
}

}  // extern "C"
