// gbin_internal.h — host-side declarations of the kernel launchers (one .cu per stage).
// Every launcher returns the number of kernels it launched (for gbin_timings.kernel_launches).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "bin3.cuh"
#include "gbin_device.cuh"

namespace gbin {

// Per-kernel-class device timing (CUDA events on the launching stream), for the roofline numbers
// bench.py reports.  Disabled by default; when disabled begin/end cost one branch.
enum KernelKind { KK_SCAN = 0, KK_RADIX_HIST, KK_RADIX_TILESCAN, KK_RADIX_SCATTER, KK_RUNS, KK_PRUNE, KK_EMIT, KK_SKR_SCAN, KK_SKR_PLAN, KK_SKR_GROUP, KK_V3_ENTRIES, KK_V3_SPAN, KK_COUNT };
struct KernelProf {
    static constexpr int MAX_REGIONS = 256;
    bool enabled = false;
    bool created = false;
    int n = 0;
    cudaEvent_t a[MAX_REGIONS], b[MAX_REGIONS];
    unsigned char kind[MAX_REGIONS];
    float ms[KK_COUNT];
    unsigned launches[KK_COUNT];
    void reset() {
        n = 0;
        for (int i = 0; i < KK_COUNT; i++) { ms[i] = 0.f; launches[i] = 0; }
    }
    bool begin(int k, cudaStream_t st) {
        if (!enabled || n >= MAX_REGIONS) return false;
        if (!created) {
            for (int i = 0; i < MAX_REGIONS; i++) { cudaEventCreate(&a[i]); cudaEventCreate(&b[i]); }
            created = true;
        }
        kind[n] = (unsigned char)k;
        cudaEventRecord(a[n], st);
        return true;
    }
    void end(bool on, int nlaunch, cudaStream_t st) {
        if (!on) return;
        cudaEventRecord(b[n], st);
        launches[kind[n]] += (unsigned)nlaunch;
        n++;
    }
    void collect() {  // call after the stream is synchronised
        for (int i = 0; i < n; i++) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, a[i], b[i]) == cudaSuccess) ms[kind[i]] += t;
            else (void)cudaGetLastError();
        }
        n = 0;
    }
    void destroy() {
        if (created) for (int i = 0; i < MAX_REGIONS; i++) { cudaEventDestroy(a[i]); cudaEventDestroy(b[i]); }
        created = false;
    }
};

// ---- scan_reads.cu
int launch_count_windows(const ReadsView &rv, int K, uint32_t *counts, cudaStream_t st);
int launch_scan_reads(const ReadsView &rv, const uint64_t *rec_off, int K, int M, int KW, uint32_t arrival_base, uint32_t max_len,
                      void *out, unsigned long long *bad_bases, int sm_count, cudaStream_t st);
uint32_t scan_reads_max_len();

// ---- radix_sort.cu
// Stable LSD radix sort of n records by (mmer, kmer) ascending.  The result lands in `a` or `b`;
// the function returns which through *result_in_b.  tile_hist: scratch of radix_scratch_bytes(n).
size_t radix_scratch_bytes(uint64_t n);
int radix_sort_records(void *a, void *b, uint64_t n, int KW, int K, int M, void *scratch, bool *result_in_b, int *passes_out,
                       KernelProf *prof, cudaStream_t st);
// Stable partition by owner = owner_of_mmer(mmer, n_parts): in -> out, part sizes to d_counts[n_parts] (device, u64).
int radix_partition_by_owner(const void *in, void *out, uint64_t n, int KW, uint32_t n_parts, void *scratch, uint64_t *d_counts,
                             cudaStream_t st);

// Owner exchange over peer memory (one process per GPU, CUDA IPC; see radix_sort.cu).
constexpr int XCHG_MAX_WORLD = 16;
struct XchgShared {  // one per rank, in device memory, mapped by every peer
    unsigned long long counts[XCHG_MAX_WORLD * XCHG_MAX_WORLD];  // counts[s * XCHG_MAX_WORLD + d]: records rank s sends to owner d (row s written by rank s)
    unsigned int count_flag[XCHG_MAX_WORLD];                     // epoch of rank s's row
    unsigned int done_flag[XCHG_MAX_WORLD];                      // epoch: rank s has finished storing into this rank's receive buffer
};
struct XchgResult {  // device scalars of the last exchange
    unsigned long long n_in;                  // records received
    unsigned long long sent[XCHG_MAX_WORLD];  // records sent per owner
    unsigned int status;                      // 0 ok, 1 an owner's receive buffer is too small (nothing was stored), 2 a peer did not answer
    unsigned int pad;
};
struct XchgPlan {  // passed to the kernels by value
    uint32_t rank, world, epoch, pad;
    XchgShared *peer_sh[XCHG_MAX_WORLD];   // [rank] = own
    void *peer_recv[XCHG_MAX_WORLD];       // receive buffers
    unsigned long long cap[XCHG_MAX_WORLD];  // their capacities in records
    char **dst_tab;                        // device, [XCHG_MAX_WORLD]: per-owner destinations of this exchange
    XchgResult *result;                    // device
    long long timeout_cycles;              // how long a kernel waits for a peer's flag (0: the default below)
};
int radix_exchange_skr_by_owner(const void *in, uint64_t n, int skr_words, void *scratch, const XchgPlan &xp, cudaStream_t st);

// v2: super-k-mer records (skr.cuh), sorted / partitioned on their m-mer code (word 1).
// side_out (n u64, optional): {m-mer code << 32 | windows} of every record in sorted order, written by the last pass.
int radix_sort_skr_by_mmer(void *a, void *b, uint64_t n, int skr_words, int M, void *scratch, bool *result_in_b, int *passes_out,
                           uint64_t *side_out, KernelProf *prof, cudaStream_t st);
int radix_partition_skr_by_owner(const void *in, void *out, uint64_t n, int skr_words, uint32_t n_parts, void *scratch, uint64_t *d_counts,
                                 cudaStream_t st);
// Stable select of part `part` of n_parts: the records (super-k-mer records of rec_words 8 | 12 when skr, else instance records of
// rec_words 4 | 6) with owner_of_mmer(m-mer, n_parts) == part go to out[0..) in input order; counters[0] += their number,
// counters[1] += their k-mer instances.  tile_state: select_part_state_bytes(n), ticket: one u32 (both zeroed here).
size_t select_part_state_bytes(uint64_t n);
int select_part(const void *in, uint64_t n, int rec_words, bool skr, uint32_t part, uint32_t n_parts, void *out, unsigned long long *tile_state,
                uint32_t *ticket, unsigned long long *counters, cudaStream_t st);

// ---- skr_scan.cu
// Scans reads [read_begin, read_end) of rv; record offsets continue from counters[1] (zero it before the first launch).
int launch_skr_scan(const ReadsView &rv, uint64_t read_begin, uint64_t read_end, int K, int M, uint32_t arrival_base, uint32_t max_len,
                    void *out, uint64_t capacity, unsigned long long *tile_state, uint32_t *ticket, unsigned long long *counters, int sm_count,
                    cudaStream_t st);
uint32_t skr_scan_tiles(uint64_t n_reads, int K, int M, uint32_t max_len);

// ---- skr_group.cu (pipeline v2: plan units, group in shared memory, emit)
struct SkrGroupCounters {  // mirror of GroupCounters in skr_group.cu
    unsigned long long distinct;
    unsigned long long total_kmers, total_ids;
    unsigned int overflow, ticket, n_units, n_big, big_inst, pad[3];
};
size_t skr_group_smem_bytes(int KW);
uint64_t skr_max_units(uint64_t n_inst, uint64_t n_runs);
uint64_t skr_max_big_runs(uint64_t n_inst);
int skr_plan_runs(const uint64_t *side, uint64_t n_skr, uint32_t *inst_prefix, uint64_t *both64, uint32_t *run_start,
                  uint64_t *scratch64, uint32_t *n_inst_dev, uint32_t *n_runs_dev, cudaStream_t st);
size_t skr_unit_bytes();
int skr_plan_units(const void *skr_sorted, int K, const uint32_t *inst_prefix, const uint32_t *run_start, uint64_t n_runs,
                   uint32_t *small_prefix, uint32_t *unit_base, uint32_t *scratch, void *units, uint64_t max_units, void *gc_dev,
                   uint32_t *big_list, uint64_t *big_k0, uint64_t *big_k1, uint32_t *big_arr, int sm_count, cudaStream_t st);
// The grouping runs as ch.n consecutive launches over equal ranges of the unit list, one chained scan across them.
// With totals_dev set, the end offsets of every chunk ({k-mers << 31 | ids}) are published after it (and copied to
// totals_host / followed by the event done[c] when those are given), so the host can stream finished parts of the table.
constexpr int SKR_MAX_CHUNKS = 16;
struct SkrGroupChunks {
    uint32_t n;                       // 1..SKR_MAX_CHUNKS
    uint32_t *tickets;                // device, [n], zeroed by the launcher
    unsigned long long *totals_dev;   // device, [n] or nullptr
    unsigned long long *totals_host;  // pinned, [n] or nullptr
    cudaEvent_t *done;                // [n] or nullptr
};
int skr_group_launch(const void *skr_sorted, int K, int cutoff, const uint32_t *inst_prefix, const void *units, unsigned long long *unit_state,
                     uint64_t max_units, const SkrGroupChunks &ch, void *gc_dev, uint64_t *big_k0, uint64_t *big_k1, uint32_t *big_arr, const int32_t *ids_by_arrival, int32_t id_base, uint64_t *kmer_codes,
                     uint32_t *kmer_mmer, uint64_t *kmer_id_off, int32_t *read_ids, uint64_t kmer_cap, uint64_t id_cap, int32_t *stg_ids, uint64_t *stg_codes,
                     uint32_t *stg_mmer, uint32_t *stg_off, int sm_count, cudaStream_t st);
int skr_emit_buckets(const uint32_t *kmer_mmer, uint64_t n_kmers, uint64_t n_ids, uint32_t *bucket_excl, uint32_t *scratch,
                     uint32_t *mmer_codes, uint64_t *mmer_kmer_off, uint64_t *kmer_id_off, uint32_t *n_buckets_dev, cudaStream_t st);

// ---- bin3.cu (pipeline v3: sort by reference, one warp or one pair of warps per unit, table written once at its final place)
// slot_info (per slot) is gathered into sorted_info (per sorted entry) by the last pass
int radix_sort_entries(void *a, void *b, uint64_t n, int key_bits, void *scratch, bool *result_in_b, int *passes_out, const uint16_t *slot_info,
                       uint16_t *sorted_info, KernelProf *prof, cudaStream_t st, const unsigned long long *n_real_dev = nullptr);
int expand_ids_device(const uint64_t *id_off, const int32_t *ids, uint64_t n_kmers, uint32_t K, uint64_t *list_off, int32_t *exp_ids, int sm_count,
                      cudaStream_t st);
int v3_make_entries(const void *skr, uint64_t n_rec, const KeyLayout &kl, uint64_t *ent, uint16_t *piece_info, unsigned long long *n_real_dev,
                    cudaStream_t st);
int v3_plan_runs(const uint64_t *ent, const uint16_t *sorted_info, uint64_t n_ent, uint32_t *inst_prefix, uint64_t *both64, uint32_t *run_start,
                 uint64_t *scratch64, uint32_t *n_inst_dev, uint32_t *n_runs_dev, cudaStream_t st);
uint64_t v3_max_units(uint64_t n_inst, uint64_t n_runs, int cap);
size_t v3_unit_bytes();
size_t v3_unit_out_bytes();
struct V3Counters {  // mirror of G3Counters in bin3.cu
    unsigned long long distinct, total_kmers, total_ids;
    unsigned int overflow, n_units, n_spans, pad;
    unsigned long long lsd_kmers, lsd_ids;
};
int v3_plan_units(const uint16_t *sorted_info, const uint64_t *ent, const KeyLayout &kl, int cap, const uint32_t *inst_prefix, const uint32_t *run_start, uint64_t n_runs,
                  uint64_t *nunits64, uint64_t *base64, uint32_t *atom3, uint32_t *spanlen, uint32_t *head_run, void *scratch, void *units, uint64_t max_units,
                  void *gc_dev, uint32_t n_chunks, uint32_t *chunk_bounds, cudaStream_t st);
struct V3Out {
    // the flat table
    uint64_t *kmer_codes;
    uint32_t *kmer_mmer;
    uint64_t *kmer_id_off;
    int32_t *read_ids;
    // staging (unit-local places) and what every unit reports
    uint64_t kmer_cap, id_cap;
    uint64_t *stg_codes;
    uint32_t *stg_mmer;
    uint32_t *stg_loff;
    int32_t *stg_ids;
    void *unit_out;
    uint64_t id_off_base;  // ids emitted by earlier passes of the batch
};
struct V3Lsd {  // arrays of the global sort that puts long spans in order (cap = 0: none allocated)
    void *rec;
    uint32_t *src_off, *cnt, *fidx, *nadj;
    uint64_t cap;
};
struct V3Chunks {
    uint32_t n;                       // 1..SKR_MAX_CHUNKS launches over consecutive ranges of the unit list
    uint32_t *tickets;                // device, [2 * n], zeroed by the launcher
    uint32_t *bounds;                 // device, [n + 1], filled by v3_plan_units
    uint64_t *chunk_sum;              // device scalar (scratch)
    unsigned long long *totals_dev;   // device, [n]: {k-mers << 32 | ids} emitted up to the end of every chunk
    unsigned long long *lsd_totals_dev;  // device, [n]: the same for the k-mers handed to the global sort
    unsigned long long *totals_host, *lsd_totals_host;  // pinned, [n] or nullptr
    cudaEvent_t *done;                // [n] or nullptr
    cudaStream_t aux;                 // second stream + two events (no timing): the two grouping launches of a chunk run side by side
    cudaEvent_t ev_fork, ev_join;
};
size_t v3_group_smem_bytes(int KW, int cap);
int v3_group_launch(const void *skr, const uint64_t *ent, const void *units, const KeyLayout &kl, int cap, int cutoff, const int32_t *ids_by_arrival, int32_t id_base,
                    const V3Out &o, uint64_t max_units, uint64_t *unit_excl, uint64_t *lsd_excl, void *scan_scratch, void *gc_dev, const V3Chunks &ch, const V3Lsd &lsd,
                    bool finalize_only, int sm_count, KernelProf *prof, cudaStream_t st);
int v3_lsd_finish(const KeyLayout &kl, uint64_t n, void *rec_a, void *rec_b, void *radix_scratch, uint64_t *dnew, void *scan_scratch, const V3Out &o, const V3Lsd &lsd,
                  int sm_count, KernelProf *prof, cudaStream_t st);
uint32_t v3_pass_tiles(uint64_t n_ent);
uint32_t v3_pass_tile_entries();
int v3_pass_tile_sums(const uint16_t *sorted_info, uint64_t n_ent, unsigned long long *sums_dev, cudaStream_t st);
int v3_pass_bounds(const uint64_t *ent, uint64_t n_ent, int mshift, unsigned long long *bounds_dev, uint32_t n_bounds, cudaStream_t st);
size_t v3_mmer_bitmap_bytes(int M);
int v3_count_mmers(const void *skr, int skr_words, uint64_t n_rec, int M, uint32_t *bitmap, unsigned long long *count_dev, cudaStream_t st);

// ---- table_digest.cu
}  // namespace gbin
struct gbin_table;
namespace gbin {
int table_digest_device(const ::gbin_table *t, unsigned long long *out_dev, cudaStream_t st);
uint64_t table_digest_host(const ::gbin_table *t);

// ---- split_reads.cu (main's fgets loop on the device)
uint32_t split_tiles(uint64_t n);
int split_find_newlines(const uint8_t *data, uint64_t n, uint32_t *tile_counts, uint32_t *scan_scratch, uint64_t *nl, uint32_t *n_nl_dev,
                        bool emit, cudaStream_t st);
int split_count_reads(const uint64_t *nl, uint64_t n_nl, uint64_t size, uint32_t cap, uint64_t n_lines, uint32_t *read_base, uint32_t *scan_scratch,
                      uint32_t *n_reads_dev, cudaStream_t st);
int split_emit_reads(const uint64_t *nl, uint64_t n_nl, uint64_t size, uint32_t cap, uint64_t n_lines, const uint32_t *read_base, uint64_t *starts,
                     uint32_t *lens, cudaStream_t st);

// ---- group_prune.cu
struct GroupCounts {  // device-resident scalars, copied to the host between phases
    uint32_t n_distinct, n_kmers, n_buckets, pad;
    uint64_t n_ids;
};
struct GroupWorkspace {  // all device pointers, sized by the caller (capi.cu)
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
size_t group_scan_scratch_bytes(uint64_t n);
// Phase 1: run-length over sorted records -> group_of, run_start, counts->n_distinct.
int group_find_runs(const void *sorted, uint64_t n, int KW, GroupWorkspace &ws, cudaStream_t st);
// Phase 2 (needs n_distinct on the host): prune decision + offsets -> counts->n_kmers, n_ids.
int group_prune_offsets(uint64_t n, uint64_t n_distinct, int cutoff, GroupWorkspace &ws, cudaStream_t st);
// Phase 3 (needs n_kmers on the host): bucket boundaries over surviving k-mers -> counts->n_buckets.
int group_mark_buckets(const void *sorted, int KW, uint64_t n_distinct, uint64_t n_kmers, GroupWorkspace &ws, cudaStream_t st);
// Phase 4: emit the flat table.
struct TableOut {
    uint32_t *mmer_codes;
    uint64_t *mmer_kmer_off;
    uint64_t *kmer_codes;
    uint64_t *kmer_id_off;
    int32_t *read_ids;
};
int group_emit(const void *sorted, uint64_t n, int KW, uint64_t n_distinct, uint64_t n_kmers, uint64_t n_ids, uint64_t n_buckets,
               const int32_t *ids_by_arrival, int32_t id_base, GroupWorkspace &ws, const TableOut &out, cudaStream_t st);

}  // namespace gbin
