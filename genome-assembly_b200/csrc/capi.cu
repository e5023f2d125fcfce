// capi.cu — the extern "C" layer of libgbin.so: the context, read checks and staging, the scan stage and the fallback ladder
// (pipeline 3 -> 2 -> 1), the host calls, the owner parts path, the owner exchange and the multi-GPU call.
// The grouping pipelines keep their host orchestration next to their kernels: run_v3_group (bin3.cu), run_v2_group
// (skr_group.cu), run_group (group_prune.cu).
// There is no CPU fallback anywhere in this file: every entry point either runs the CUDA kernels or
// returns an error code.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "gbin_ctx.h"
#include "prefix_scan.cuh"

using namespace gbin;

namespace {

// Host path only: the reads are still in host memory; the scan stage copies them chunk by chunk on the copy stream and
// scans every chunk as soon as it has landed.
struct HostFeed {
    const char *src;     // host
    char *dst;           // device
    uint64_t bytes;
    int chunks;
};

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

}  // namespace

namespace gbin {

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

}  // namespace gbin

namespace {

// What was streamed into the sink belongs to an abandoned attempt: wait until nothing is in flight into the arenas, then start over.
int abandon_sink(gbin_ctx *ctx, HostSink *sink) {
    if (!sink) return GBIN_OK;
    CU(cudaStreamSynchronize(ctx->st_d2h));
    sink->kmers_done = sink->ids_done = 0;
    return GBIN_OK;
}

// The big arrays of a host table are streamed into the pinned arenas as far as these reach (they are sized by the previous call,
// so the first call on a context copies everything at the end and later calls of similar size overlap the copy).
HostSink host_sink(gbin_ctx *ctx) {
    HostSink sink{static_cast<uint64_t *>(ctx->h_kmer_codes.p), static_cast<uint64_t *>(ctx->h_kmer_id_off.p), static_cast<int32_t *>(ctx->h_read_ids.p),
                  0, 0, 0, 0, ctx->host_chunks};
    sink.kmer_cap = ctx->h_kmer_codes.cap / (sizeof(uint64_t) * ctx->KW);
    if (ctx->h_kmer_id_off.cap / sizeof(uint64_t) < sink.kmer_cap) sink.kmer_cap = ctx->h_kmer_id_off.cap / sizeof(uint64_t);
    sink.id_cap = ctx->h_read_ids.cap / sizeof(int32_t);
    return sink;
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

// The checks of a reads descriptor, made before anything is copied or launched.  Reads in host memory must lie inside data_bytes and,
// when max_read_len is given, be no longer than it; ragged reads in device memory are not looked at.  *max_len (when given) receives
// the longest ragged host read.
int check_reads(gbin_ctx *ctx, const gbin_reads *rd, bool on_host, uint32_t *max_len = nullptr) {
    const uint64_t n = rd->n_reads, bytes = rd->data_bytes;
    if (n == 0) return GBIN_OK;
    if (!rd->data) return fail(ctx, GBIN_E_INVALID_ARG, "reads->data is NULL");
    if (n >= (1ull << 32)) return fail(ctx, GBIN_E_TOO_LARGE, "more than 2^32-1 reads in one batch");
    if (on_host && bytes == 0) return fail(ctx, GBIN_E_INVALID_ARG, "host reads need data_bytes");
    if (!rd->starts) {
        if (rd->stride < rd->read_len) return fail(ctx, GBIN_E_INVALID_ARG, "stride < read_len");
        if (bytes && (rd->read_len > bytes || (n > 1 && rd->stride > (bytes - rd->read_len) / (n - 1))))
            return fail(ctx, GBIN_E_INVALID_ARG, "fixed-stride reads exceed data_bytes");
        return GBIN_OK;
    }
    if (!rd->lens) return fail(ctx, GBIN_E_INVALID_ARG, "ragged reads need lens");
    uint32_t mx = 0;
    for (uint64_t i = 0; on_host && i < n; i++) {
        const uint64_t s = rd->starts[i], len = rd->lens[i];
        if (s > bytes || len > bytes - s) return fail(ctx, GBIN_E_INVALID_ARG, "read %llu exceeds data_bytes", (unsigned long long)i);
        if (rd->max_read_len && len > rd->max_read_len) return fail(ctx, GBIN_E_INVALID_ARG, "read %llu is longer than max_read_len", (unsigned long long)i);
        if (len > mx) mx = (uint32_t)len;
    }
    if (max_len) *max_len = mx;
    return GBIN_OK;
}

ReadsView reads_view(const gbin_reads *rd) {
    return ReadsView{reinterpret_cast<const uint8_t *>(rd->data), rd->data_bytes, rd->n_reads, rd->stride, rd->read_len, rd->starts, rd->lens};
}

// Reads [r0, r1) of a batch, which span bytes [b0, b1) of its data.
struct ReadRange {
    uint64_t r0, r1, b0, b1;
    uint32_t max_len;  // 0: not known on the host (plan_reads finds it)
};

// The range [r0, r1) (r0 < r1) of a checked descriptor, with its byte span and longest read: one pass over it for ragged reads.
ReadRange read_range(const gbin_reads *rd, uint64_t r0, uint64_t r1) {
    if (!rd->starts) return {r0, r1, r0 * rd->stride, (r1 - 1) * rd->stride + rd->read_len, rd->read_len};
    uint64_t b0 = ~0ull, b1 = 0;
    uint32_t ml = 0;
    for (uint64_t i = r0; i < r1; i++) {
        const uint64_t s = rd->starts[i], e = s + rd->lens[i];
        if (s < b0) b0 = s;
        if (e > b1) b1 = e;
        if (rd->lens[i] > ml) ml = rd->lens[i];
    }
    return {r0, r1, b0, b1, ml ? ml : 1};
}

// Enqueues on `st` the copy of the host reads of `r` into staging slot `slot` and makes *view the device batch of those reads (its
// read 0 is read r.r0; no ids).  Ragged starts are rebased to r.b0 in the slot's pinned array, or copied as they are when r.b0 == 0.
// The slot must be free: whatever read it before has finished.  The caller records its own events around the copy.
int stage_host_reads(gbin_ctx *ctx, const gbin_reads *rd, const ReadRange &r, int slot, cudaStream_t st, gbin_reads *view) {
    ReadStage &s = ctx->stage[slot];
    const uint64_t m = r.r1 - r.r0, bytes = r.b1 - r.b0;
    *view = *rd;
    view->n_reads = m;
    view->read_ids = nullptr;
    view->max_read_len = r.max_len;
    CU(s.data.ensure(bytes + 64));
    if (bytes) CU(cudaMemcpyAsync(s.data.p, rd->data + r.b0, bytes, cudaMemcpyHostToDevice, st));
    view->data = s.data.as<char>();
    view->data_bytes = bytes;
    if (!rd->starts) return GBIN_OK;
    const uint64_t *starts = rd->starts + r.r0;
    if (r.b0) {
        CU(s.rebased.ensure(m * sizeof(uint64_t)));
        uint64_t *rebased = static_cast<uint64_t *>(s.rebased.p);
        for (uint64_t i = 0; i < m; i++) rebased[i] = starts[i] - r.b0;
        starts = rebased;
    }
    CU(s.meta.ensure(m * (sizeof(uint64_t) + sizeof(uint32_t)) + 16));
    CU(cudaMemcpyAsync(s.meta.p, starts, m * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(s.meta.as<char>() + m * sizeof(uint64_t), rd->lens + r.r0, m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    view->starts = s.meta.as<uint64_t>();
    view->lens = reinterpret_cast<const uint32_t *>(s.meta.as<char>() + m * sizeof(uint64_t));
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

// Finds the instance count and the longest read of a descriptor in device memory that check_reads passed or the library built, and
// refuses reads longer than gbin_max_read_len().
// On return: *n_inst, *max_len, and for the ragged form ctx->rec_off holds per-read record offsets.
int plan_reads(gbin_ctx *ctx, const gbin_reads *rd, cudaStream_t st, uint64_t *n_inst, uint32_t *max_len, int *launches) {
    const int K = ctx->cfg.kmer_size;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    *n_inst = 0;
    *max_len = 0;
    if (rd->n_reads == 0) return GBIN_OK;
    if (!rd->starts) {
        *max_len = rd->read_len;
        *n_inst = rd->read_len >= (uint32_t)K ? rd->n_reads * (uint64_t)(rd->read_len - K + 1) : 0;
    } else {
        CU(ctx->win_counts.ensure(rd->n_reads * sizeof(uint32_t)));
        CU(ctx->rec_off.ensure((rd->n_reads + 1) * sizeof(uint64_t)));
        CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(rd->n_reads)));
        CU(cudaMemsetAsync(&dm->reads.max_len, 0, sizeof(unsigned int), st));
        if (rd->max_read_len == 0) {
            max_len_kernel<<<(unsigned)((rd->n_reads + 255) / 256), 256, 0, st>>>(rd->lens, rd->n_reads, &dm->reads.max_len);
            (*launches)++;
        }
        *launches += launch_count_windows(reads_view(rd), K, ctx->win_counts.as<uint32_t>(), st);
        *launches += exclusive_scan<uint64_t, WinCountIn>(WinCountIn{ctx->win_counts.as<uint32_t>()}, ctx->rec_off.as<uint64_t>(), rd->n_reads,
                                                          ctx->scan_scratch.as<uint64_t>(),
                                                          reinterpret_cast<uint64_t *>(&dm->reads.total_windows), st);
        CU(read_back(ctx, &Misc::reads, st));
        *n_inst = hm->reads.total_windows;
        *max_len = rd->max_read_len ? rd->max_read_len : hm->reads.max_len;
    }
    if (*max_len > gbin_max_read_len()) return fail(ctx, GBIN_E_TOO_LARGE, "read length %u exceeds the limit of %u bases", *max_len, gbin_max_read_len());
    return GBIN_OK;
}

int run_scan(gbin_ctx *ctx, const gbin_reads *rd, uint32_t arrival_base, void *d_records, uint32_t max_len, cudaStream_t st, int *launches) {
    Misc *dm = ctx->misc.as<Misc>();
    CU(cudaMemsetAsync(&dm->grp.bad_bases, 0, sizeof(unsigned long long), st));
    const bool on = ctx->prof.begin(KK_SCAN, st);
    const int ls = launch_scan_reads(reads_view(rd), rd->starts ? ctx->rec_off.as<uint64_t>() : nullptr, ctx->cfg.kmer_size, ctx->cfg.mmer_size, ctx->KW,
                                     arrival_base, max_len ? max_len : 1, d_records, &dm->grp.bad_bases, ctx->sm_count, st);
    ctx->prof.end(on, ls < 0 ? 0 : ls, st);
    if (ls < 0) return fail(ctx, GBIN_E_TOO_LARGE, "a read of %u bases does not fit the scan kernel's shared memory (limit %u bases)", max_len, gbin_max_read_len());
    *launches += ls;
    CU(cudaGetLastError());
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
            const int l1 = launch_skr_scan(reads_view(rd), r0, r1, K, M, arrival_base, max_len, ext ? ext : ctx->skr_a.p, cap, ctx->tile_state.as<unsigned long long>(),
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
    for (int i = 0; i < 4 && e == cudaSuccess; i++) e = cudaEventCreate(&ctx->ev_part_h2d[i]);
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
    for (int i = 0; i < 4; i++) cudaEventDestroy(ctx->ev_part_h2d[i]);
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
    } else if (!strcmp(name, "part_chunk_kb")) {
        if (value < 1) return GBIN_E_INVALID_ARG;
        ctx->part_chunk_bytes = (uint64_t)value << 10;
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
    int rc = check_reads(ctx, reads, false);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int launches = 0;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    rc = bin_device_impl(ctx, reads, st, out, &launches);
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

// The end of a host call, after `rc` from its device stage: on success the table goes to the pinned arenas and the call's timings are
// taken; on failure the copy streams are drained, so that no copy into or out of the context's buffers outlives the call.
static int finish_host_call(gbin_ctx *ctx, int rc, const gbin_table &dev, HostSink *sink, cudaStream_t st, int launches, gbin_table *out) {
    if (rc) {
        cudaStreamSynchronize(ctx->st_h2d);
        cudaStreamSynchronize(ctx->st_d2h);
        return rc;
    }
    rc = table_to_pinned(ctx, dev, sink, st, out);
    if (rc) return rc;
    CU(cudaEventRecord(ctx->ev[EV_TABLE_ON_HOST], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaStreamSynchronize(ctx->st_d2h));
    finish_timings(ctx, launches, true);
    return GBIN_OK;
}

int gbin_bin_reads_host(gbin_ctx *ctx, const gbin_reads *reads, gbin_table *out) {
    if (!ctx || !reads || !out) return GBIN_E_INVALID_ARG;
    uint32_t max_len = 0;
    int rc = check_reads(ctx, reads, true, &max_len);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, nullptr, &st));
    int launches = 0;
    const uint64_t n = reads->n_reads;
    gbin_reads d = *reads;
    HostFeed feed{};
    const bool use_feed = n && !reads->starts;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    if (use_feed) {
        // fixed stride: read ranges are byte ranges, so the copy is left to the scan stage, which overlaps it with the scan
        CU(ctx->stage[0].data.ensure(reads->data_bytes + 64));
        d.data = ctx->stage[0].data.as<char>();
        feed = HostFeed{reads->data, ctx->stage[0].data.as<char>(), reads->data_bytes, ctx->host_chunks};
        if (n < 4096u * (uint64_t)feed.chunks) feed.chunks = 1;
        CU(cudaStreamWaitEvent(ctx->st_h2d, ctx->ev[EV_START], 0));
    } else if (n) {  // ragged: the whole buffer, and the longest read known on the host spares the device reduction
        const ReadRange all{0, n, 0, reads->data_bytes, reads->max_read_len ? reads->max_read_len : (max_len ? max_len : 1)};
        if ((rc = stage_host_reads(ctx, reads, all, 0, st, &d))) return rc;
    }
    if (n && reads->read_ids) {
        CU(ctx->d_ids.ensure(n * sizeof(int32_t)));
        CU(cudaMemcpyAsync(ctx->d_ids.p, reads->read_ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        d.read_ids = ctx->d_ids.as<int32_t>();
    }
    if (!use_feed) CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    HostSink sink = host_sink(ctx);
    gbin_table dev;
    rc = bin_device_impl(ctx, &d, st, &dev, &launches, use_feed ? &feed : nullptr, &sink);
    return finish_host_call(ctx, rc, dev, &sink, st, launches, out);
}

// ---------------------------------------------------------------- the table in owner parts, one part per call

namespace {
// Cuts the reads into chunks of whole reads whose byte span is at most ctx->part_chunk_bytes, with at least one read each.
// Fixed-stride reads: contiguous byte ranges.  Ragged reads in host memory: the span [min start, max end) of the chunk's reads, which
// is copied whole and exceeds the budget only for a single read longer than it (the chunk buffer then grows to fit).  Reads laid out
// out of order make more, shorter chunks.
// Ragged reads in device memory are scanned where they are, so they are cut by read count, at the mean bytes per read.
std::vector<ReadRange> plan_part_chunks(const gbin_ctx *ctx, const gbin_reads *rd, bool on_host) {
    const uint64_t n = rd->n_reads, budget = ctx->part_chunk_bytes;
    std::vector<ReadRange> out;
    if (n == 0) return out;
    if (!rd->starts || !on_host) {
        const uint64_t per_read = rd->starts ? rd->data_bytes / n + 1 : rd->stride;
        const uint64_t per = per_read == 0 ? n : (budget / per_read ? budget / per_read : 1);
        for (uint64_t r0 = 0; r0 < n; r0 += per) {
            const uint64_t r1 = n - r0 > per ? r0 + per : n;
            out.push_back(rd->starts ? ReadRange{r0, r1, 0, rd->data_bytes, rd->max_read_len} : read_range(rd, r0, r1));
        }
        return out;
    }
    for (uint64_t r0 = 0, r1; r0 < n; r0 = r1) {
        uint64_t lo = rd->starts[r0], hi = lo + rd->lens[r0];
        uint32_t ml = rd->lens[r0];
        for (r1 = r0 + 1; r1 < n; r1++) {
            const uint64_t s = rd->starts[r1], e = s + rd->lens[r1];
            const uint64_t nlo = s < lo ? s : lo, nhi = e > hi ? e : hi;
            if (nhi - nlo > budget) break;
            lo = nlo;
            hi = nhi;
            if (rd->lens[r1] > ml) ml = rd->lens[r1];
        }
        out.push_back({r0, r1, lo, hi, ml ? ml : 1});
    }
    return out;
}

// Streams every chunk through the device and keeps the records of part `part` in ctx->part_rec, in arrival order: super-k-mer
// records, or instance records when `inst`.  Host form: chunk c is copied into slot c & 1 on the copy stream while chunk c - 1 is
// scanned; the slot's previous chunk has been scanned and selected by then (the host waited for both).  *too_long: the
// super-k-mer scan cannot hold these reads, nothing was selected.  *scan_ms / *h2d_ms: scan + select / copy time summed over chunks.
int scan_select_part(gbin_ctx *ctx, const gbin_reads *rd, bool on_host, const std::vector<ReadRange> &chunks, uint32_t part, uint32_t n_parts,
                     bool inst, cudaStream_t st, int *launches, uint64_t *n_sel, uint64_t *n_sel_inst, bool *too_long, float *scan_ms, float *h2d_ms) {
    const int words = inst ? 2 * ctx->KW + 2 : (ctx->cfg.kmer_size <= 32 ? 8 : 12);
    const size_t rb = 4u * (size_t)words;
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    *n_sel = *n_sel_inst = 0;
    *too_long = false;
    CU(cudaMemsetAsync(dm->part_sel, 0, sizeof dm->part_sel, st));
    gbin_reads staged[2];  // the chunks in the two staging slots
    auto copy_in = [&](size_t c) -> int {
        const int s = (int)(c & 1);
        CU(cudaEventRecord(ctx->ev_part_h2d[2 * s], ctx->st_h2d));
        if (const int rc = stage_host_reads(ctx, rd, chunks[c], s, ctx->st_h2d, &staged[s])) return rc;
        CU(cudaEventRecord(ctx->ev_part_h2d[2 * s + 1], ctx->st_h2d));
        return GBIN_OK;
    };
    auto elapsed = [](cudaEvent_t a, cudaEvent_t b) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, a, b) != cudaSuccess) (void)cudaGetLastError();
        return t;
    };
    int rc = (on_host && !chunks.empty()) ? copy_in(0) : GBIN_OK;
    for (size_t c = 0; !rc && c < chunks.size(); c++) {
        const ReadRange &k = chunks[c];
        const int s = (int)(c & 1);
        if (on_host && c + 1 < chunks.size() && (rc = copy_in(c + 1))) return rc;
        gbin_reads v = *rd;  // the chunk as a batch of its own, scanned with arrival_base = its first read
        v.n_reads = k.r1 - k.r0;
        v.read_ids = nullptr;
        v.max_read_len = k.max_len;
        if (on_host) {
            v = staged[s];
            CU(cudaStreamWaitEvent(st, ctx->ev_part_h2d[2 * s + 1], 0));
        } else if (rd->starts) {
            v.starts = rd->starts + k.r0;
            v.lens = rd->lens + k.r0;
        } else {
            v.data = rd->data + k.b0;
            v.data_bytes = k.b1 - k.b0;
        }
        CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
        uint64_t n_c = 0, n_src = 0;
        uint32_t max_len = 0;
        if ((rc = plan_reads(ctx, &v, st, &n_c, &max_len, launches))) return rc;
        const void *src = nullptr;
        if (n_c && inst) {
            CU(ctx->rec_b.ensure((n_c + 1) * rb));
            if ((rc = run_scan(ctx, &v, (uint32_t)k.r0, ctx->rec_b.p, max_len, st, launches))) return rc;
            CU(read_back(ctx, &Misc::grp, st));
            if (hm->grp.bad_bases) return fail(ctx, GBIN_E_NON_ACGT, "%llu bases other than A/C/G/T in the batch", hm->grp.bad_bases);
            src = ctx->rec_b.p;
            n_src = n_c;
        } else if (n_c) {
            rc = run_skr_scan(ctx, &v, n_c, max_len, (uint32_t)k.r0, nullptr, 0, st, &n_src, launches);
            if (rc == GBIN_E_TOO_LARGE) {  // reads longer than the super-k-mer scan holds in shared memory
                *too_long = true;
                return GBIN_OK;
            }
            if (rc) return rc;
            src = ctx->skr_a.p;
        }
        if (n_src) {
            const uint64_t need = *n_sel + n_src;  // every record of the chunk might belong to the part
            if ((need + 1) * rb > ctx->part_rec.cap) {
                // grow towards what the whole call is expected to select: the part's records so far, extrapolated over the reads
                uint64_t want = (uint64_t)((double)(*n_sel + n_src / n_parts + 1) * (double)rd->n_reads / (double)k.r1 * 1.1);
                if (want < need) want = need;
                CU(ctx->part_rec.ensure_keep((want + 1) * rb, *n_sel * rb, st));
            }
            CU(ctx->part_state.ensure(select_part_state_bytes(n_src)));
            const bool on = ctx->prof.begin(KK_RADIX_SCATTER, st);
            const int l = select_part(src, n_src, words, !inst, part, n_parts, ctx->part_rec.as<char>() + *n_sel * rb, ctx->part_state.as<unsigned long long>(),
                                      &dm->part_ticket, dm->part_sel, st);
            ctx->prof.end(on, l, st);
            *launches += l;
            CU(cudaGetLastError());
            CU(read_back(ctx, &Misc::part_sel, st));
            *n_sel = hm->part_sel[0];
            *n_sel_inst = hm->part_sel[1];
        }
        CU(cudaEventRecord(ctx->ev[EV_SCANNED], st));
        CU(cudaEventSynchronize(ctx->ev[EV_SCANNED]));
        *scan_ms += elapsed(ctx->ev[EV_READS_ON_DEVICE], ctx->ev[EV_SCANNED]);
        if (on_host) *h2d_ms += elapsed(ctx->ev_part_h2d[2 * s], ctx->ev_part_h2d[2 * s + 1]);
    }
    return rc;
}

// One part of the table (gbin_bin_reads_host_part / gbin_bin_reads_device_part) into the context's device table.  The part is
// selected from super-k-mer records and grouped by pipeline 3 (2 when 3 gives it up); it is redone from the reads in instance-record
// form (pipeline 1) when pipeline 2 overflows too, when the reads are too long for the super-k-mer scan, or when the context is set
// to pipeline 1.  sink: the host form's pinned arenas.
int bin_part_impl(gbin_ctx *ctx, const gbin_reads *rd, bool on_host, uint32_t part, uint32_t n_parts, cudaStream_t st, HostSink *sink, gbin_table *out,
                  int *launches, float *scan_ms, float *h2d_ms) {
    if (n_parts == 0 || n_parts > 65536 || part >= n_parts) return fail(ctx, GBIN_E_INVALID_ARG, "part %u of %u parts (need part < n_parts <= 65536)", part, n_parts);
    const uint64_t n = rd->n_reads;
    const std::vector<ReadRange> chunks = plan_part_chunks(ctx, rd, on_host);
    const int32_t *d_ids = rd->read_ids;  // looked up by arrival = index over all the reads
    if (on_host && rd->read_ids && n) {
        CU(ctx->d_ids.ensure(n * sizeof(int32_t)));
        CU(cudaMemcpyAsync(ctx->d_ids.p, rd->read_ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        d_ids = ctx->d_ids.as<int32_t>();
    }
    bool inst = ctx->pipeline == 1;
    for (;;) {
        uint64_t n_sel = 0, n_sel_inst = 0;
        bool too_long = false;
        int rc = scan_select_part(ctx, rd, on_host, chunks, part, n_parts, inst, st, launches, &n_sel, &n_sel_inst, &too_long, scan_ms, h2d_ms);
        CU(cudaStreamSynchronize(ctx->st_h2d));  // a copy into a chunk buffer may still be in flight when the loop ended early
        if (rc) return rc;
        if (too_long) {
            ctx->fallbacks++;
            inst = true;
            continue;
        }
        if (!inst && n_sel) {
            // the chunks' record buffer is dead: lend it to pipeline 3's entry sort, as gbin_donate_scratch does
            ctx->donated = ctx->skr_a.p;
            ctx->donated_bytes = ctx->skr_a.cap;
            bool done = false;
            int used = 2;
            uint64_t n_chk = 0;
            rc = run_skr_group(ctx, ctx->part_rec.p, n_sel, d_ids, rd->id_base, st, out, launches, &done, &n_chk, sink, &used);
            ctx->donated = nullptr;
            ctx->donated_bytes = 0;
            if (rc) return rc;
            if (done) {
                if (n_chk != n_sel_inst)
                    return fail(ctx, GBIN_E_CUDA, "internal: the part's records hold %llu windows, grouped %llu", (unsigned long long)n_sel_inst, (unsigned long long)n_chk);
                ctx->last_pipeline = used;
                break;
            }
            if ((rc = abandon_sink(ctx, sink))) return rc;
            inst = true;  // a shared-memory unit overflowed: this part goes through pipeline 1
            continue;
        }
        // instance records (or an empty part): sort + run-length + prune + emit in HBM
        if (n_sel >= (1ull << 32) - 8192) return fail(ctx, GBIN_E_TOO_LARGE, "%llu k-mer instances in one part: too many for pipeline 1", (unsigned long long)n_sel);
        memset(&ctx->rs, 0, sizeof ctx->rs);
        CU(ctx->rec_b.ensure((n_sel + 1) * (sizeof(uint64_t) * ctx->KW + 8)));
        CU(cudaMemsetAsync(&ctx->misc.as<Misc>()->grp.bad_bases, 0, sizeof(unsigned long long), st));
        rc = run_group(ctx, n_sel ? ctx->part_rec.p : nullptr, ctx->rec_b.p, n_sel, d_ids, rd->id_base, st, out, launches, ctx->ev[EV_SORTED]);
        if (rc) return rc;
        ctx->last_pipeline = inst ? 1 : ctx->pipeline;
        break;
    }
    CU(cudaEventRecord(ctx->ev[EV_GROUPED], st));
    return GBIN_OK;
}

// gbin_plan_parts' model of a part call's device memory (DESIGN.md §5).  PART_BYTES_PER_INSTANCE per k-mer instance of the part: the
// largest high-water mark per instance measured on a B200 for a one-part call (57.1 B at the config-5 shape; configs 2, 4 and the
// config-3 shape 46.4 / 56.6 / 53.9 B) — its records, pipeline 3's sort, plan, staging and table with the buffers' slack, and there
// also the read chunk.  PART_SKEW: the owner hash's imbalance (1.4 % for the busiest of 8 owners, DESIGN.md §6) with room for larger
// P.  PART_BYTES_PER_CHUNK_BYTE per byte of part_chunk_kb: two read chunks + one chunk's super-k-mer records, which the scan sizes at
// a quarter of the chunk's instances (+ reads) x 32 B with 1/16 slack: 2 + 0.8 x 0.25 x 32 x 17/16 ~ 9 for 150-base reads.
constexpr double PART_BYTES_PER_INSTANCE = 58.0, PART_SKEW = 1.05, PART_BYTES_PER_CHUNK_BYTE = 9.0;
}  // namespace

int gbin_bin_reads_host_part(gbin_ctx *ctx, const gbin_reads *reads, uint32_t part, uint32_t n_parts, gbin_table *out) {
    if (!ctx || !reads || !out) return GBIN_E_INVALID_ARG;
    int rc = check_reads(ctx, reads, true);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, nullptr, &st));
    int launches = 0;
    float scan_ms = 0.f, h2d_ms = 0.f;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    HostSink sink = host_sink(ctx);
    gbin_table dev;
    rc = bin_part_impl(ctx, reads, true, part, n_parts, st, &sink, &dev, &launches, &scan_ms, &h2d_ms);
    if ((rc = finish_host_call(ctx, rc, dev, &sink, st, launches, out))) return rc;
    ctx->tm.h2d_ms = h2d_ms;
    ctx->tm.scan_ms = scan_ms;
    return GBIN_OK;
}

int gbin_bin_reads_device_part(gbin_ctx *ctx, const gbin_reads *reads, uint32_t part, uint32_t n_parts, void *stream, gbin_table *out) {
    if (!ctx || !reads || !out) return GBIN_E_INVALID_ARG;
    int rc = check_reads(ctx, reads, false);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    int launches = 0;
    float scan_ms = 0.f, h2d_ms = 0.f;
    CU(cudaEventRecord(ctx->ev[EV_START], st));
    rc = bin_part_impl(ctx, reads, false, part, n_parts, st, nullptr, out, &launches, &scan_ms, &h2d_ms);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    finish_timings(ctx, launches, false);
    ctx->tm.scan_ms = scan_ms;
    return GBIN_OK;
}

int gbin_plan_parts(gbin_ctx *ctx, uint64_t n_instances, uint32_t *n_parts_out) {
    if (!ctx || !n_parts_out) return GBIN_E_INVALID_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    const double room = (double)free_b - PART_BYTES_PER_CHUNK_BYTE * (double)ctx->part_chunk_bytes;
    auto fits = [&](uint64_t P) { return PART_BYTES_PER_INSTANCE * PART_SKEW * (double)((n_instances + P - 1) / P) <= room; };
    const double est = room > 0 ? PART_BYTES_PER_INSTANCE * PART_SKEW * (double)n_instances / room : 65537.0;
    uint64_t P = est < 65537.0 ? (uint64_t)est : 65537;
    if (P < 1) P = 1;
    while (P > 1 && fits(P - 1)) P--;
    while (P <= 65536 && !fits(P)) P++;
    if (P > 65536)
        return fail(ctx, GBIN_E_NOMEM, "%llu k-mer instances do not fit %llu free bytes in 65536 parts", (unsigned long long)n_instances, (unsigned long long)free_b);
    *n_parts_out = (uint32_t)P;
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
    CU(ctx->stage[0].meta.ensure((n_reads + 1) * (sizeof(uint64_t) + sizeof(uint32_t))));
    uint64_t *starts = ctx->stage[0].meta.as<uint64_t>();
    uint32_t *lens = reinterpret_cast<uint32_t *>(starts + n_reads + 1);
    *launches += split_emit_reads(ctx->split_nl.as<uint64_t>(), n_nl, size, cap, n_lines, ctx->split_base.as<uint32_t>(), starts, lens, st);
    CU(cudaGetLastError());
    out->n_reads = n_reads;
    out->starts = starts;
    out->lens = lens;
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
    if (e == cudaSuccess) e = ctx->stage[0].data.ensure(size + 64);
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
    if (size) CU(cudaMemcpyAsync(ctx->stage[0].data.p, ctx->h_file.p, size, cudaMemcpyHostToDevice, st));
    CU(cudaEventRecord(ctx->ev[EV_READS_ON_DEVICE], st));
    gbin_reads rd;
    gbin_table dev;
    int rc = split_reads_impl(ctx, ctx->stage[0].data.as<char>(), size, read_length_define, st, &rd, &launches);
    if (!rc) rc = bin_device_impl(ctx, &rd, st, &dev, &launches);
    return finish_host_call(ctx, rc, dev, nullptr, st, launches, out);
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
    const int rc = check_reads(ctx, reads, false);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint32_t max_len = 0;
    int launches = 0;
    return plan_reads(ctx, reads, st, n_out, &max_len, &launches);
}

int gbin_scan_reads_device(gbin_ctx *ctx, const gbin_reads *reads, uint32_t arrival_base, void *d_records, uint64_t capacity,
                           void *stream, uint64_t *n_out) {
    if (!ctx || !reads || !n_out) return GBIN_E_INVALID_ARG;
    int rc = check_reads(ctx, reads, false);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint64_t n = 0;
    uint32_t max_len = 0;
    int launches = 0;
    if ((rc = plan_reads(ctx, reads, st, &n, &max_len, &launches))) return rc;
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
    int rc = check_reads(ctx, reads, false);
    if (rc) return rc;
    cudaStream_t st;
    CU(begin_call(ctx, stream, &st));
    uint64_t n = 0, n_skr = 0;
    uint32_t max_len = 0;
    int launches = 0;
    if ((rc = plan_reads(ctx, reads, st, &n, &max_len, &launches))) return rc;
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
    m->err[0] = 0;
    if (const int rc = check_reads(m->ctx[0], reads, true)) {
        snprintf(m->err, sizeof m->err, "%s", gbin_last_error(m->ctx[0]));
        return rc;
    }
    const int G = m->n;
    const uint64_t n = reads->n_reads;
    std::vector<int> rcs(G, GBIN_OK);
    std::vector<uint64_t> n_skr(G, 0);
    std::vector<uint64_t> part_counts((size_t)G * G, 0);  // [g * G + o]: instance records GPU g holds for owner o (overflow redo)
    std::vector<std::string> errs(G);
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
        gbin_reads d{};  // no reads when the shard is empty
        const int r0 = cnt ? stage_host_reads(ctx, reads, read_range(reads, lo, hi), 0, st, &d) : GBIN_OK;
        if (r0) failed(r0, "copying the shard to the device");
        cudaError_t e = cudaSuccess;
        const int32_t *d_ids = nullptr;
        if (!rc && reads->read_ids && n) {  // ids are looked up by global arrival index: every GPU holds the whole array
            e = ctx->d_ids.ensure(n * sizeof(int32_t));
            if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_ids.p, reads->read_ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, st);
            d_ids = ctx->d_ids.as<int32_t>();
        }
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            failed(e == cudaErrorMemoryAllocation ? GBIN_E_NOMEM : GBIN_E_CUDA, "copying the read ids to the device");
        }
        // ---- scan into this context's record buffer (sized by an estimate, regrown to the exact need when short)
        uint64_t ninst = 0, cap = 0;
        if (!rc && cnt) {
            uint64_t est = 0;
            const int r1 = gbin_count_instances_device(ctx, &d, st, &est);
            if (r1) failed(r1, "counting the instances");
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
