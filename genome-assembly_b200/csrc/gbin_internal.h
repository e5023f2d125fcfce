// gbin_internal.h — host-side declarations of what one .cu file provides to the others: kernel launchers and one entry per
// grouping pipeline.  Every launcher returns the number of kernels it launched (for gbin_timings.kernel_launches).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "bin3.cuh"
#include "gbin_device.cuh"

struct gbin_ctx;
struct gbin_table;

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

// ---- the grouping pipelines.  Each groups n_skr super-k-mer records (pipeline 1: n instance records) into the context's device
// table *out and counts its kernel launches in *launches.  Pipelines 3 and 2 set *done = false when the batch does not fit them
// (the caller falls back to the next pipeline); *n_inst_out receives the k-mer instances the records hold.  sink (host path):
// finished chunks of the table are streamed into it while later ones are grouped.
struct HostSink;
constexpr int SKR_MAX_CHUNKS = 16;  // consecutive grouping launches over the unit list, after each of which the table can be streamed

// ---- bin3.cu (pipeline 3: sort by reference, one warp or one pair of warps per unit, table written once at its final place).
// The records in `skr` are read, not moved.
int run_v3_group(gbin_ctx *ctx, const void *skr, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, ::gbin_table *out, int *launches,
                 bool *done, uint64_t *n_inst_out, HostSink *sink);
// slot_info (per slot) is gathered into sorted_info (per sorted entry) by the last pass (radix_sort.cu)
int radix_sort_entries(void *a, void *b, uint64_t n, int key_bits, void *scratch, bool *result_in_b, int *passes_out, const uint16_t *slot_info,
                       uint16_t *sorted_info, KernelProf *prof, cudaStream_t st, const unsigned long long *n_real_dev = nullptr);

// ---- skr_group.cu (pipeline 2: records sorted by m-mer, one CTA per unit).  `skr` is clobbered; `twin` is the sort's second buffer.
struct GroupCounters {  // device scalars of the grouping kernels
    unsigned long long distinct;
    unsigned long long total_kmers, total_ids;  // written by the last unit
    unsigned int overflow;
    unsigned int ticket;
    unsigned int n_units;
    unsigned int n_big;     // buckets larger than a unit (work list of partition_big_runs_kernel)
    unsigned int big_inst;  // k-mer instances in those buckets (allocation cursor of the scratch arrays)
    unsigned int pad[3];
};
int run_v2_group(gbin_ctx *ctx, void *skr, void *twin, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, ::gbin_table *out,
                 int *launches, bool *done, uint64_t *n_inst_out, HostSink *sink);

// ---- expand_ids.cu
int expand_ids_device(const uint64_t *id_off, const int32_t *ids, uint64_t n_kmers, uint32_t K, uint64_t *list_off, int32_t *exp_ids, int sm_count,
                      cudaStream_t st);

// ---- table_digest.cu
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
size_t group_scan_scratch_bytes(uint64_t n);  // scratch of the prefix scans (prefix_scan.cuh) over n elements
// Sort + run-length + prune + emit of n instance records living in `recs` (scratch twin `twin`); ev_sorted (optional) is recorded after the sort.
int run_group(gbin_ctx *ctx, void *recs, void *twin, uint64_t n, const int32_t *d_ids, int32_t id_base, cudaStream_t st, ::gbin_table *out,
              int *launches, cudaEvent_t ev_sorted);

}  // namespace gbin
