// gbin_ctx.h — the context behind the C ABI (struct gbin_ctx) and the host helpers that capi.cu and the three grouping pipelines
// (group_prune.cu, skr_group.cu, bin3.cu) share: device and pinned buffers, the device scalars and their read-back, error reporting.
#pragma once
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/gbin.h"
#include "gbin_internal.h"

namespace gbin {

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

// A range of host reads copied to the device (stage_host_reads): its bytes, its starts (rebased to the first copied byte) followed by
// its lens, and the pinned host array the starts are rebased in.  Slot 0 also holds gbin_bin_file_host's file image and its split.
struct ReadStage {
    DevBuf data, meta;
    HostBuf rebased;
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
    GroupCounters gc;
    uint32_t chunk_tickets[SKR_MAX_CHUNKS];
    // pipeline 3
    G3Counters gc3;
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
    // one owner part per call: records and k-mer instances selected so far, and the select kernel's ticket
    unsigned long long part_sel[2];
    uint32_t part_ticket;
};

// Host path only: pinned destinations for the big arrays of the table; finished chunks of the grouping are copied out on the
// second copy stream while later chunks are still running.
struct HostSink {
    uint64_t *kmer_codes, *kmer_id_off;  // pinned; capacities in k-mers
    int32_t *read_ids;                   // pinned; capacity in ids
    uint64_t kmer_cap, id_cap;
    uint64_t kmers_done, ids_done;       // what has been enqueued for copy so far
    int chunks;
};

// Timing events of one call, in the order they are recorded.
enum : int { EV_START, EV_READS_ON_DEVICE, EV_SCANNED, EV_SORTED, EV_GROUPED, EV_TABLE_ON_HOST, EV_COUNT };

}  // namespace gbin

struct gbin_ctx {
    gbin_config cfg;
    int KW;
    int sm_count;
    cudaStream_t stream;
    cudaStream_t st_h2d, st_d2h;  // copy streams of the host path (H2D of later read chunks / D2H of finished table chunks overlap the kernels)
    cudaEvent_t ev_feed[gbin::SKR_MAX_CHUNKS], ev_chunk[gbin::SKR_MAX_CHUNKS], ev_copy;
    cudaStream_t st_aux;          // second compute stream of pipeline 3's grouping stage
    cudaEvent_t ev_fork, ev_join;
    int host_chunks;              // GBIN_HOST_CHUNKS (default 8; 1 = no overlap)
    char err[512];
    gbin_timings tm;
    cudaEvent_t ev[gbin::EV_COUNT];
    // inputs staged by the host path: [0] a whole batch or shard, or a chunk of the parts path, which alternates with [1]
    gbin::ReadStage stage[2];
    gbin::DevBuf d_ids;
    // pipeline workspace
    gbin::DevBuf rec_a, rec_b, radix_scratch, win_counts, rec_off, scan_scratch;
    gbin::DevBuf group_of, run_start, surv_index, id_offset, surv_group, bucket_of;
    gbin::DevBuf misc;
    // workspace of the super-k-mer pipelines (2 and 3)
    gbin::DevBuf skr_a, skr_b, tile_state, inst_prefix, run_excl, skr_run_start, small_prefix, unit_base, units, unit_state, o_kmer_mmer, bucket_excl, big_list, big_k0, big_k1, big_arr, stg_ids, stg_codes, stg_mmer, stg_off, skr_side;
    // pipeline 3 workspace
    gbin::DevBuf ent_a, ent_b, piece_n, sorted_info, v3_base64, v3_head_run, v3_unit_out, v3_unit_excl, v3_atoms, v3_lsd_aux, v3_bitmap;
    gbin::DevBuf x_list_off, x_ids;         // gbin_expand_read_ids_device's result
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
        gbin::XchgShared *sh = nullptr;
        char **dst_tab = nullptr;
        gbin::XchgResult *result = nullptr;
        gbin::XchgPlan plan;
        void *opened[2 * gbin::XCHG_MAX_WORLD];
        int n_opened = 0;
    } xg;
    // device-resident result
    gbin::DevBuf o_mmer_codes, o_mmer_kmer_off, o_kmer_codes, o_kmer_id_off, o_read_ids;
    // pinned host arena for results of the host path + small readbacks
    gbin::HostBuf h_misc, h_result, h_kmer_codes, h_kmer_id_off, h_read_ids, h_file;
    gbin::DevBuf split_nl, split_tiles_buf, split_base;  // device-side fgets splitting
    // one owner part per call: the part's records, the select's tiles
    gbin::DevBuf part_rec, part_state;
    uint64_t part_chunk_bytes = 1ull << 30;  // gbin_set_tuning "part_chunk_kb"
    cudaEvent_t ev_part_h2d[4];              // [2 * slot + 0 | 1]: around the copy of a chunk into slot 0 | 1 (timed)
    gbin::KernelProf prof;
};

namespace gbin {

inline int fail(gbin_ctx *ctx, int code, const char *fmt, ...) {
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

// Copies one member of the device scalars into the pinned mirror and waits for it: one host round trip.
template <typename T>
cudaError_t read_back(gbin_ctx *ctx, T Misc::*field, cudaStream_t st) {
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    const cudaError_t e = cudaMemcpyAsync(&(hm->*field), &(dm->*field), sizeof(T), cudaMemcpyDeviceToHost, st);
    return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
}

// The device table over the context's output arrays.
inline gbin_table device_table(const gbin_ctx *ctx, uint64_t n_instances, uint64_t n_distinct, uint64_t S, uint64_t NS, uint64_t B) {
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

// Host path: streams the finished part of the table to the host while later chunks are grouped (capi.cu).  The table is written in
// unit order, and what the units of chunk c wrote is final once ctx->ev_chunk[c] has fired; totals_host[c] then holds
// {k-mers << shift | ids} written up to the end of chunk c.  A chunk with k-mers left to pipeline 3's global sort for long spans
// (lsd_totals_host[c] != 0) ends the streaming, as does an arena too small: the rest is copied at the end.
int stream_finished_chunks(gbin_ctx *ctx, HostSink *sink, uint32_t n, const unsigned long long *totals_host, int shift,
                           const unsigned long long *lsd_totals_host);
// Bucket directory of the super-k-mer pipelines over the S surviving k-mers in ctx->o_kmer_mmer; *B receives the bucket count
// (skr_group.cu).
int emit_bucket_directory(gbin_ctx *ctx, uint64_t S, uint64_t NS, cudaStream_t st, int *launches, uint64_t *B);

}  // namespace gbin
