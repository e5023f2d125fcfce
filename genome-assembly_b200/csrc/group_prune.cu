// group_prune.cu — run-length, prune and emit over the sorted records.
//
// What the reference does per k-mer with pointer structures becomes segmented array passes:
//   * one group per distinct (m-mer, k-mer)          — the level-2 zhash entry (binning.c:1052-1058)
//   * group length                                   — the ll_node list length that prune_kmers
//                                                      counts (binning.c:1094-1100)
//   * keep iff length > ABUNDANCE_CUTOFF             — binning.c:1102
//   * m-mer buckets that still own a k-mer           — prune_data drops emptied buckets (:1136-1142)
//   * ids of a group, newest arrival first           — the list walked from its head (:1059-1069)
#include "gbin_ctx.h"
#include "gbin_device.cuh"
#include "prefix_scan.cuh"

namespace gbin {

struct GroupWorkspace {  // all device pointers, sized by run_group
    uint32_t *group_of;     // [n]    group index of every sorted record
    uint32_t *run_start;    // [n+1]  first record of every group (+ sentinel n)
    uint32_t *surv_index;   // [n_distinct+1] exclusive count of surviving groups
    uint64_t *id_offset;    // [n_distinct+1] exclusive sum of surviving run lengths
    uint32_t *surv_group;   // [n_kmers] group index of surviving k-mer s
    uint32_t *bucket_of;    // [n_kmers] bucket index of surviving k-mer s
    void *scan_scratch;     // prefix-scan scratch (u64 elements)
    GroupCounts *counts;    // device
    int cutoff;             // ABUNDANCE_CUTOFF (binning.c:12); < 0 keeps everything
};
struct TableOut {
    uint32_t *mmer_codes;
    uint64_t *mmer_kmer_off;
    uint64_t *kmer_codes;
    uint64_t *kmer_id_off;
    int32_t *read_ids;
};

template <int KW>
struct HeadFlag {
    const Rec<KW> *rec;
    __device__ __forceinline__ uint32_t operator()(uint64_t j) const {
        if (j == 0) return 1u;
        return same_key<KW>(load_rec<KW>(rec + j), load_rec<KW>(rec + j - 1)) ? 0u : 1u;
    }
};

template <int KW>
__global__ void assign_groups_kernel(const Rec<KW> *__restrict__ rec, uint64_t n, uint32_t *__restrict__ group_of,
                                     uint32_t *__restrict__ run_start) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t head = HeadFlag<KW>{rec}(j);
    const uint32_t g = group_of[j] + head - 1;  // group_of holds the exclusive head count on entry
    group_of[j] = g;
    if (head) run_start[g] = (uint32_t)j;
    if (j == n - 1) run_start[g + 1] = (uint32_t)n;
}

struct SurvFlag {
    const uint32_t *run_start;
    int cutoff;
    __device__ __forceinline__ uint32_t operator()(uint64_t g) const {
        const uint32_t len = run_start[g + 1] - run_start[g];
        return (cutoff < 0 || len > (uint32_t)cutoff) ? 1u : 0u;
    }
};
struct SurvLen {
    const uint32_t *run_start;
    int cutoff;
    __device__ __forceinline__ uint64_t operator()(uint64_t g) const {
        const uint32_t len = run_start[g + 1] - run_start[g];
        return (cutoff < 0 || len > (uint32_t)cutoff) ? (uint64_t)len : 0ull;
    }
};

__global__ void compact_survivors_kernel(const uint32_t *__restrict__ run_start, const uint32_t *__restrict__ surv_index, int cutoff,
                                         uint64_t n_distinct, uint32_t *__restrict__ surv_group) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_distinct) return;
    if (SurvFlag{run_start, cutoff}(g)) surv_group[surv_index[g]] = (uint32_t)g;
}

template <int KW>
struct BucketHead {
    const Rec<KW> *rec;
    const uint32_t *run_start;
    const uint32_t *surv_group;
    __device__ __forceinline__ uint32_t operator()(uint64_t s) const {
        if (s == 0) return 1u;
        return rec[run_start[surv_group[s]]].mmer != rec[run_start[surv_group[s - 1]]].mmer ? 1u : 0u;
    }
};

template <int KW>
__global__ void emit_kmers_kernel(const Rec<KW> *__restrict__ rec, const uint32_t *__restrict__ run_start,
                                  const uint32_t *__restrict__ surv_group, const uint32_t *__restrict__ bucket_excl,
                                  const uint64_t *__restrict__ id_offset, uint64_t n_kmers, uint64_t n_ids, uint64_t n_buckets,
                                  TableOut out) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_kmers) return;
    const uint32_t g = surv_group[s];
    const Rec<KW> r = load_rec<KW>(rec + run_start[g]);
#pragma unroll
    for (int w = 0; w < KW; w++) out.kmer_codes[s * KW + w] = r.k[w];
    out.kmer_id_off[s] = id_offset[g];
    const uint32_t head = BucketHead<KW>{rec, run_start, surv_group}(s);
    if (head) {
        const uint32_t b = bucket_excl[s];
        out.mmer_codes[b] = r.mmer;
        out.mmer_kmer_off[b] = s;
    }
    if (s == n_kmers - 1) {
        out.kmer_id_off[n_kmers] = n_ids;
        out.mmer_kmer_off[n_buckets] = n_kmers;
    }
}

template <int KW>
__global__ void emit_ids_kernel(const Rec<KW> *__restrict__ rec, uint64_t n, const uint32_t *__restrict__ group_of,
                                const uint32_t *__restrict__ run_start, const uint64_t *__restrict__ id_offset, int cutoff,
                                const int32_t *__restrict__ ids_by_arrival, int32_t id_base, int32_t *__restrict__ read_ids) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t g = group_of[j];
    const uint32_t j0 = run_start[g], len = run_start[g + 1] - j0;
    if (!(cutoff < 0 || len > (uint32_t)cutoff)) return;
    const uint32_t arrival = rec[j].arrival;
    // records of a group are in arrival order (stable sort); the list is read newest first
    const uint64_t pos = id_offset[g] + (len - 1 - ((uint32_t)j - j0));
    read_ids[pos] = ids_by_arrival ? ids_by_arrival[arrival] : id_base + (int32_t)arrival;
}

__global__ void empty_table_kernel(TableOut out) {
    out.kmer_id_off[0] = 0;
    out.mmer_kmer_off[0] = 0;
}

size_t group_scan_scratch_bytes(uint64_t n) { return (scan_scratch_elems(n ? n : 1) + 8) * sizeof(uint64_t); }

static inline unsigned blocks_for(uint64_t n) { return (unsigned)((n + 255) / 256); }

// Phase 1: run-length over sorted records -> group_of, run_start, counts->n_distinct.
static int group_find_runs(const void *sorted, uint64_t n, int KW, GroupWorkspace &ws, cudaStream_t st) {
    if (n == 0) {
        cudaMemsetAsync(ws.counts, 0, sizeof(GroupCounts), st);
        return 0;
    }
    int launches = 0;
    uint32_t *tot = &ws.counts->n_distinct;
    if (KW == 1) {
        const Rec<1> *r = static_cast<const Rec<1> *>(sorted);
        launches += exclusive_scan<uint32_t, HeadFlag<1>>(HeadFlag<1>{r}, ws.group_of, n, static_cast<uint32_t *>(ws.scan_scratch), tot, st);
        assign_groups_kernel<1><<<blocks_for(n), 256, 0, st>>>(r, n, ws.group_of, ws.run_start);
    } else {
        const Rec<2> *r = static_cast<const Rec<2> *>(sorted);
        launches += exclusive_scan<uint32_t, HeadFlag<2>>(HeadFlag<2>{r}, ws.group_of, n, static_cast<uint32_t *>(ws.scan_scratch), tot, st);
        assign_groups_kernel<2><<<blocks_for(n), 256, 0, st>>>(r, n, ws.group_of, ws.run_start);
    }
    return launches + 1;
}

// Phase 2 (needs n_distinct on the host): prune decision + offsets -> counts->n_kmers, n_ids.
static int group_prune_offsets(uint64_t n, uint64_t n_distinct, int cutoff, GroupWorkspace &ws, cudaStream_t st) {
    (void)n;
    int launches = 0;
    launches += exclusive_scan<uint32_t, SurvFlag>(SurvFlag{ws.run_start, cutoff}, ws.surv_index, n_distinct,
                                                   static_cast<uint32_t *>(ws.scan_scratch), &ws.counts->n_kmers, st);
    launches += exclusive_scan<uint64_t, SurvLen>(SurvLen{ws.run_start, cutoff}, ws.id_offset, n_distinct,
                                                  static_cast<uint64_t *>(ws.scan_scratch), &ws.counts->n_ids, st);
    return launches;
}

// Phase 3 (needs n_kmers on the host): bucket boundaries over surviving k-mers -> counts->n_buckets.
static int group_mark_buckets(const void *sorted, int KW, uint64_t n_distinct, uint64_t n_kmers, GroupWorkspace &ws, cudaStream_t st) {
    if (n_kmers == 0) {
        cudaMemsetAsync(&ws.counts->n_buckets, 0, sizeof(uint32_t), st);
        return 0;
    }
    int launches = 1;
    compact_survivors_kernel<<<blocks_for(n_distinct), 256, 0, st>>>(ws.run_start, ws.surv_index, ws.cutoff, n_distinct, ws.surv_group);
    if (KW == 1)
        launches += exclusive_scan<uint32_t, BucketHead<1>>(BucketHead<1>{static_cast<const Rec<1> *>(sorted), ws.run_start, ws.surv_group},
                                                            ws.bucket_of, n_kmers, static_cast<uint32_t *>(ws.scan_scratch),
                                                            &ws.counts->n_buckets, st);
    else
        launches += exclusive_scan<uint32_t, BucketHead<2>>(BucketHead<2>{static_cast<const Rec<2> *>(sorted), ws.run_start, ws.surv_group},
                                                            ws.bucket_of, n_kmers, static_cast<uint32_t *>(ws.scan_scratch),
                                                            &ws.counts->n_buckets, st);
    return launches;
}

// Phase 4: emit the flat table.
static int group_emit(const void *sorted, uint64_t n, int KW, uint64_t n_distinct, uint64_t n_kmers, uint64_t n_ids, uint64_t n_buckets,
               const int32_t *ids_by_arrival, int32_t id_base, GroupWorkspace &ws, const TableOut &out, cudaStream_t st) {
    (void)n_distinct;
    if (n_kmers == 0) {
        empty_table_kernel<<<1, 1, 0, st>>>(out);
        return 1;
    }
    if (KW == 1) {
        const Rec<1> *r = static_cast<const Rec<1> *>(sorted);
        emit_kmers_kernel<1><<<blocks_for(n_kmers), 256, 0, st>>>(r, ws.run_start, ws.surv_group, ws.bucket_of, ws.id_offset, n_kmers, n_ids,
                                                                n_buckets, out);
        emit_ids_kernel<1><<<blocks_for(n), 256, 0, st>>>(r, n, ws.group_of, ws.run_start, ws.id_offset, ws.cutoff, ids_by_arrival, id_base,
                                                         out.read_ids);
    } else {
        const Rec<2> *r = static_cast<const Rec<2> *>(sorted);
        emit_kmers_kernel<2><<<blocks_for(n_kmers), 256, 0, st>>>(r, ws.run_start, ws.surv_group, ws.bucket_of, ws.id_offset, n_kmers, n_ids,
                                                                n_buckets, out);
        emit_ids_kernel<2><<<blocks_for(n), 256, 0, st>>>(r, n, ws.group_of, ws.run_start, ws.id_offset, ws.cutoff, ids_by_arrival, id_base,
                                                         out.read_ids);
    }
    return 2;
}

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

}  // namespace gbin
