/*
 * gbin.h — C ABI of libgbin.so: the B200-native k-mer binning hot path of twitu/genome-assembly.
 *
 * The reference has no plugin/FFI layer; its boundary is the plain C function surface of binning.c
 * (SURVEY.md §8b).  libgbin.so therefore exports
 *   (1) the reference's own entry points for this path, same names and argument meaning:
 *         process_read  (binning.c:902)   prune_data (binning.c:1130)
 *         getval        (binning.c:91)    getbp      (binning.c:69)     getscore (binning.c:114)
 *       operating on the reference's own struct ZHashTable / ZHashEntry / ll_node layouts
 *       (zhash.h:14-26, llist.h:7-13; restated in gbin_ref_types.h), and
 *   (2) the batch / device entry points below (gbin_*), which are the fast path the shims call.
 *
 * Everything is extern "C", plain pointers and sizes; no CUDA or torch types appear in signatures
 * (streams are passed as void*, i.e. a cudaStream_t).  Errors are returned as negative ints — the
 * library never calls exit() (the reference's zmalloc does, zhash.c:230-250).
 *
 * Contract differences from the reference, all deliberate and documented in DESIGN.md:
 *   - K, M and the cutoff are runtime values (reference: #defines at binning.c:10-13).
 *     Supported: 2 <= M <= 15, 2M <= K <= 64 (for K < 2M the reference's else-branch loop at
 *     binning.c:997 is live and scores overflow; every BASELINE config has K >= 2M).
 *   - Reads must consist of A/C/G/T only; any other byte makes the call fail with
 *     GBIN_E_NON_ACGT (the reference would keep the raw byte inside un-flipped keys,
 *     binning.c:1023-1026, which a 2-bit code cannot represent).
 *   - The result is a flat table in canonical order (m-mer code ascending, k-mer code ascending,
 *     read ids newest-first) instead of a pointer graph whose iteration order depends on hash
 *     layout; gbin_table_to_zhash() materialises the reference's pointer graph when a consumer
 *     needs it.
 */
#ifndef GBIN_H
#define GBIN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBIN_OK 0
#define GBIN_E_INVALID_CONFIG (-1) /* K/M/cutoff outside the supported range */
#define GBIN_E_CUDA (-2)           /* a CUDA call failed; see gbin_last_error() */
#define GBIN_E_NOMEM (-3)
#define GBIN_E_NON_ACGT (-4)       /* a read holds a byte other than A, C, G, T */
#define GBIN_E_STATE (-5)          /* call sequence error (e.g. process_read after prune_data) */
#define GBIN_E_TOO_LARGE (-6)      /* batch exceeds an implementation limit (see DESIGN.md) */
#define GBIN_E_INVALID_ARG (-7)
#define GBIN_E_IO (-8)

#define GBIN_MAX_READ_LEN 4096
/* Longest read a batch may hold on this device: min(GBIN_MAX_READ_LEN, what one warp's shared memory holds).  Reads of more than
 * about 1800 bases are scanned by pipeline 1's kernel (the super-k-mer scan keeps more per read in shared memory). */
uint32_t gbin_max_read_len(void);

/* Runtime form of binning.c:10-12. */
typedef struct gbin_config {
    int32_t kmer_size;        /* KMER_SIZE        (binning.c:11) */
    int32_t mmer_size;        /* MMER_SIZE        (binning.c:10) */
    int32_t abundance_cutoff; /* ABUNDANCE_CUTOFF (binning.c:12): keep a k-mer iff its list length > cutoff; < 0 disables the prune */
    int32_t device;           /* CUDA device ordinal */
} gbin_config;

/* The pruned two-level store mmer_hash -> kmer_hash -> read-id list (binning.c:1044-1069 after
 * prune_data), flattened.  All codes are base-4 with T,G,C,A = 0..3 (getval, binning.c:91-111) and
 * the first character most significant, i.e. getscore() of the key string (binning.c:114-124).
 *   bucket b  : m-mer mmer_codes[b], owns k-mers [mmer_kmer_off[b], mmer_kmer_off[b+1])
 *   k-mer  s  : code kmer_codes[s*kmer_words .. ] (most significant word first),
 *               owns read ids [kmer_id_off[s], kmer_id_off[s+1]) — newest first, exactly the order
 *               in which the reference's linked list is walked from its head (binning.c:1059-1069).
 * Buckets ascend by m-mer code; k-mers ascend by code within a bucket. */
typedef struct gbin_table {
    int32_t kmer_size, mmer_size, abundance_cutoff;
    int32_t kmer_words;      /* 1 when K <= 32, else 2 */
    int32_t on_device;       /* 1: the pointers below are device pointers owned by the context */
    int32_t ctx_owned;       /* 1: arrays belong to the context (valid until its next call); gbin_table_free is then a no-op */
    uint64_t n_instances;    /* k-mer instances (windows) processed */
    uint64_t n_distinct;     /* distinct (m-mer, k-mer) pairs before the prune */
    uint64_t n_buckets;      /* surviving m-mer buckets */
    uint64_t n_kmers;        /* surviving k-mers */
    uint64_t n_ids;          /* read-id nodes in surviving lists */
    uint32_t *mmer_codes;    /* [n_buckets] */
    uint64_t *mmer_kmer_off; /* [n_buckets + 1] */
    uint64_t *kmer_codes;    /* [n_kmers * kmer_words] */
    uint64_t *kmer_id_off;   /* [n_kmers + 1] */
    int32_t *read_ids;       /* [n_ids] */
} gbin_table;

/* Reads are given either fixed-stride (starts == NULL: read i is reads[i*stride .. i*stride+read_len))
 * or ragged (read i is reads[starts[i] .. starts[i]+lens[i])).  Reads shorter than K yield nothing
 * but still own their arrival index / id, as in main (binning.c:1165).  read_ids == NULL means
 * id = id_base + i. Arrival order == index order.
 * Every entry point that takes reads checks the descriptor before it copies or launches anything: data != NULL, n_reads < 2^32
 * (else GBIN_E_TOO_LARGE), stride >= read_len and fixed-stride reads inside a non-zero data_bytes, lens given for ragged reads.
 * The host entry points also need data_bytes != 0 and check every ragged read against it, and enforce a non-zero max_read_len as an
 * upper bound on every lens[i]; ragged reads in device memory are trusted.  Any of these fails with GBIN_E_INVALID_ARG unless noted. */
typedef struct gbin_reads {
    const char *data;       /* ASCII bases; host or device memory depending on the entry point */
    uint64_t data_bytes;    /* bytes addressable from data */
    uint64_t n_reads;
    uint64_t stride;        /* fixed-stride form */
    uint32_t read_len;      /* fixed-stride form */
    int32_t id_base;
    const uint64_t *starts; /* ragged form (NULL for fixed stride) */
    const uint32_t *lens;
    const int32_t *read_ids; /* optional explicit ids (what process_read's read_id argument carries) */
    uint32_t max_read_len;  /* ragged form: upper bound on lens[] (0 = let the library find it; host entry points refuse a longer read) */
    uint32_t reserved;
} gbin_reads;

typedef struct gbin_ctx gbin_ctx;

/* Per-stage device times of the last gbin_bin_* call, in milliseconds (CUDA events on the call's stream). */
typedef struct gbin_timings {
    float h2d_ms, scan_ms, sort_ms, group_ms, d2h_ms, total_ms;
    uint32_t kernel_launches; /* kernels launched by the last call */
    uint32_t sort_passes;
} gbin_timings;

const char *gbin_strerror(int code);
const char *gbin_last_error(const gbin_ctx *ctx);
int gbin_version(void);

int gbin_create(const gbin_config *cfg, gbin_ctx **out);
void gbin_destroy(gbin_ctx *ctx);
int gbin_get_config(const gbin_ctx *ctx, gbin_config *out);

/* Whole hot path, HOST buffers: H2D copy of the reads, pack + window/signature scan (process_read,
 * binning.c:918-1040), grouping (the two-level zhash insert, binning.c:1044-1069), prune
 * (binning.c:1085-1144), D2H of the table into the context's pinned result arena (ctx_owned = 1:
 * valid until the next call on the context; gbin_table_clone makes an independent malloc'ed copy).
 * Fixed-stride reads are copied in GBIN_HOST_CHUNKS (default 8) pieces that are scanned as they land, and the
 * finished part of the table is copied out while the rest is still being grouped (the arena is sized by the
 * previous call, so the overlap starts with the second call of similar size on a context). */
int gbin_bin_reads_host(gbin_ctx *ctx, const gbin_reads *reads, gbin_table *out);
int gbin_table_clone(const gbin_table *host, gbin_table *out);
void gbin_table_free(gbin_table *t);
/* Page-locked host memory for read buffers handed to gbin_bin_reads_host (pageable memory works, slower). */
void *gbin_pinned_alloc(size_t bytes);
void gbin_pinned_free(void *p);

/* Same, DEVICE-resident: reads->data/starts/lens/read_ids are device pointers, the table's arrays
 * stay in HBM, owned by the context and valid until the next call on it. `stream` is a cudaStream_t
 * (NULL = the context's own stream); the call returns after the work is complete on that stream. */
int gbin_bin_reads_device(gbin_ctx *ctx, const gbin_reads *reads, void *stream, gbin_table *out);

/* Copies a device-resident table to freshly malloc'ed host arrays. */
int gbin_table_to_host(gbin_ctx *ctx, const gbin_table *dev, gbin_table *host);
/* Same into the context's page-locked result arena (ctx_owned = 1: valid until the next call on the context that
 * produces a host table) — the fast way to bring a table produced by the staged / device entry points to the host. */
int gbin_table_to_pinned(gbin_ctx *ctx, const gbin_table *dev, void *stream, gbin_table *host);

/* Order-independent 64-bit digest of a table (device or host): the sum over all surviving k-mers of a hash of (m-mer code, k-mer
 * code, read-id list in list order), modulo 2^64.  Digests of tables over disjoint bucket sets add up to the digest of their
 * union, so the owners' digests of a multi-GPU run sum to the single-GPU digest.  ctx may be NULL for a host table. */
int gbin_table_digest(gbin_ctx *ctx, const gbin_table *table, void *stream, uint64_t *digest_out);

int gbin_get_timings(const gbin_ctx *ctx, gbin_timings *out);

/* Three device pipelines produce the same table:
 *   3 (default): super-k-mer records -> entries sorted by a reference to their record -> grouping/prune/emit, one warp per
 *                unit; a batch with a (bucket, d) class larger than a unit is transparently redone by pipeline 2;
 *   2          : super-k-mer records -> stable sort by m-mer -> grouping/prune/emit in shared memory; a batch
 *                that does not fit its shared-memory units (e.g. one k-mer with thousands of instances)
 *                is transparently redone by pipeline 1;
 *   1          : expanded k-mer instance records -> stable radix sort on (m-mer, k-mer) in HBM -> run-length/prune/emit.
 * So the fallback order is 3 -> 2 -> 1.  The environment variable GBIN_PIPELINE=1|2|3 selects the pipeline at context
 * creation. */
/* Sizes of the intermediate structures of the last pipeline-2 or pipeline-3 run (0 when pipeline 1 produced the table). */
typedef struct gbin_run_stats {
    uint64_t n_super_kmers; /* records emitted by the scan stage */
    uint64_t n_mmer_runs;   /* distinct m-mer codes before the prune (level-1 buckets) */
    uint64_t n_units;       /* shared-memory work units of the grouping kernel */
    uint64_t n_lsd_kmers;   /* pipeline 3: surviving k-mers of buckets spread over more than 8 units (ordered by a global sort) */
    uint32_t key_nc, key_h; /* pipeline 3: key layout of the batch (pieces per record, flank bases in the key) */
    uint32_t n_passes;      /* pipeline 3: passes over the sorted entries (more than one above 2 * 10^9 k-mer instances) */
    uint32_t reserved;
} gbin_run_stats;
int gbin_get_run_stats(const gbin_ctx *ctx, gbin_run_stats *out);
int gbin_set_pipeline(gbin_ctx *ctx, int pipeline);
/* Tuning knobs (tests and experiments; every setting produces the same table):
 *   "v3_cap" 0|512|1024    k-mer instances per work unit of pipeline 3 (default 0: 1024 with plain m-mer keys and one-word k-mers, else 512)
 *   "v3_nc"  0|1|2         pieces per super-k-mer record: 1 = key is the m-mer code; 2 = windows split by the signature's offset
 *                          and the key extended by v3_h bases next to the signature; 0 (default) = chosen per batch from the mean bucket size
 *   "v3_h"   0..           with v3_nc = 2: bases next to the signature that extend the level-1 key (clamped to what K, M allow)
 *   "v3_pass_max" >= 1000  k-mer instances per pass of pipeline 3 (default 2 * 10^9; small values exercise the multi-pass path)
 *   "xchg_timeout_ms" >= 100  how long the multi-GPU exchange kernels wait for a peer before they give up (default 120000)
 *   "host_chunks" 1..16    pieces in which gbin_bin_reads_host streams reads in / the table out
 *   "part_chunk_kb" >= 1   byte span of the read chunks of gbin_bin_reads_*_part, in KiB (default 1048576 = 1 GiB) */
int gbin_set_tuning(gbin_ctx *ctx, const char *name, int value);
/* Lends `bytes` of device memory (16-byte aligned, caller-owned) to the NEXT grouping call on the context (gbin_group_skr_device,
 * gbin_bin_reads_device): pipeline 3 puts the two buffers of its entry sort there when they fit, instead of allocating them.  The
 * memory must stay valid and unused by the caller until that call returns; the loan ends with it.  The multi-GPU path lends the scan's
 * record buffer, which is dead once the exchange has sent the records away. */
int gbin_donate_scratch(gbin_ctx *ctx, void *d_ptr, uint64_t bytes);
int gbin_get_pipeline_info(const gbin_ctx *ctx, int *configured, int *last_used, uint32_t *fallbacks);

/* Optional per-kernel-class device timing (CUDA events around each launch on the call's stream),
 * accumulated over calls since it was enabled; what bench.py's roofline line is computed from. */
#define GBIN_KERNEL_KINDS 12
typedef struct gbin_kernel_profile {
    float ms[GBIN_KERNEL_KINDS];          /* accumulated device time per kernel class */
    uint32_t launches[GBIN_KERNEL_KINDS]; /* kernels launched per class */
} gbin_kernel_profile;
int gbin_set_kernel_profiling(gbin_ctx *ctx, int enable); /* also resets the accumulators */
int gbin_get_kernel_profile(const gbin_ctx *ctx, gbin_kernel_profile *out);
const char *gbin_kernel_kind_name(int kind); /* "" past the last kind */

/* ---- staged device entry points (multi-GPU path: scan -> partition by owner -> exchange -> group) ---- */

/* Bytes per k-mer instance record produced by the scan stage (16 when K <= 32, 24 otherwise).
 * Layout: { u64 kmer words (most significant first) ; u32 mmer_code ; u32 arrival }. */
uint32_t gbin_record_bytes(const gbin_ctx *ctx);
/* Number of k-mer instances the reads will produce (reads in device memory). */
int gbin_count_instances_device(gbin_ctx *ctx, const gbin_reads *reads, void *stream, uint64_t *n_out);
/* process_read's window/signature stage for every read: writes n records in arrival order to
 * d_records (capacity in records).  arrival = arrival_base + read index. */
int gbin_scan_reads_device(gbin_ctx *ctx, const gbin_reads *reads, uint32_t arrival_base, void *d_records,
                           uint64_t capacity, void *stream, uint64_t *n_out);
/* Owner of an m-mer bucket among n_parts GPUs (SURVEY.md §8e): a multiplicative hash of the code, range-reduced
 * ((code * 0x9E3779B1 mod 2^32) * n_parts) >> 32 — the plain remainder follows the skewed last bases of the signatures. */
uint32_t gbin_owner_of(uint32_t mmer_code, uint32_t n_parts);
/* Stable partition of records by owner = gbin_owner_of(mmer_code, n_parts) into d_out;
 * counts_host[p] receives the number of records of part p (parts are laid out in order). */
int gbin_partition_records_device(gbin_ctx *ctx, const void *d_records, uint64_t n, uint32_t n_parts, void *d_out,
                                  void *stream, uint64_t *counts_host);
/* Grouping + prune of n records that are already in arrival order (d_records is used as sort
 * scratch and is clobbered).  ids: device array mapping arrival -> read id, or NULL for id_base+arrival. */
int gbin_group_records_device(gbin_ctx *ctx, void *d_records, uint64_t n, const int32_t *d_ids_by_arrival,
                              int32_t id_base, void *stream, gbin_table *out);

/* Super-k-mer form of the staged path (pipeline 2): one record per signature segment — consecutive windows that
 * keep one signature (binning.c:922) are one substring of K+n-1 bases.  Record layout (u32 words): arrival, m-mer
 * code, n | is_rev << 8, first window index, then the bases 2 bits each MSB-first (4 words for K <= 32, else 8);
 * 32 or 48 bytes.  About 1/5 of the bytes of the instance records for the same reads. */
uint32_t gbin_skr_record_bytes(const gbin_ctx *ctx);
int gbin_scan_skr_device(gbin_ctx *ctx, const gbin_reads *reads, uint32_t arrival_base, void *d_skr, uint64_t capacity, void *stream,
                         uint64_t *n_skr_out, uint64_t *n_instances_out);
int gbin_partition_skr_device(gbin_ctx *ctx, const void *d_skr, uint64_t n, uint32_t n_parts, void *d_out, void *stream,
                              uint64_t *counts_host);
/* Grouping + prune of n_skr records in arrival order (d_skr is clobbered). Fails with GBIN_E_STATE and
 * *used_fallback = 1 when a shared-memory unit overflows (degenerate inputs); the caller then re-runs the batch
 * through gbin_scan_reads_device / gbin_group_records_device. */
int gbin_group_skr_device(gbin_ctx *ctx, void *d_skr, uint64_t n_skr, const int32_t *d_ids_by_arrival, int32_t id_base, void *stream,
                          gbin_table *out, int *used_fallback);

/* ---- owner exchange over peer memory (one process per GPU on one node) ----
 * The partition by owner = gbin_owner_of(mmer_code, world) (SURVEY.md 8e) and the all-to-all are one step: every rank maps every
 * peer's receive buffer (CUDA IPC) and the partition kernel stores each owner's records straight into that owner's buffer
 * over NVLink, behind the records of the lower ranks (so arrival order is kept); counts and completion are exchanged
 * through flags in peer memory.  Setup: every rank calls gbin_xchg_create, the GBIN_XCHG_HANDLE_BYTES blobs are gathered
 * by the caller (any transport) into rank order and handed to gbin_xchg_attach on every rank.
 * gbin_xchg_exchange_skr is collective: every rank of the world must call it once per step, on contexts attached to each
 * other.  It returns this rank's receive buffer (owned by the context, valid until the next exchange) and record count;
 * GBIN_E_TOO_LARGE means some owner's buffer was too small — nothing was stored anywhere and every rank gets the same
 * error, so the caller can fall back to another transport for the step. */
#define GBIN_XCHG_HANDLE_BYTES 192
int gbin_xchg_create(gbin_ctx *ctx, uint32_t rank, uint32_t world, uint64_t capacity_records, void *handle_out);
int gbin_xchg_attach(gbin_ctx *ctx, const void *all_handles);
int gbin_xchg_exchange_skr(gbin_ctx *ctx, const void *d_skr, uint64_t n, void *stream, void **d_recv_out, uint64_t *n_recv_out,
                           uint64_t *sent_counts);
/* Teardown is collective and has two phases: every rank calls gbin_xchg_detach (closes its mappings of the peers' buffers), the
 * caller barriers, then every rank calls gbin_xchg_destroy (frees what it exported).  gbin_xchg_destroy alone detaches first, which
 * is only safe when the peers have already detached (or are gone). */
void gbin_xchg_detach(gbin_ctx *ctx);
void gbin_xchg_destroy(gbin_ctx *ctx);

/* ---- several GPUs of one node behind one C call (one process, one host thread per GPU; no Python, no MPI, no NCCL) ----
 * gbin_multi_create makes one context per device (devices == NULL: 0 .. n_devices-1) and enables peer access between them.
 * gbin_multi_bin_reads_host: reads in HOST memory; GPU g takes the contiguous read range [g*n/G, (g+1)*n/G), runs the scan, sends
 * every record to the owner of its m-mer bucket (gbin_owner_of; peer stores over NVLink, gbin_xchg_* with the peers' buffers passed
 * by address), groups what it received.  tables_out[g] (host arrays in context g's pinned arena, valid until the next call) is the
 * part of the table GPU g owns: disjoint m-mer buckets, together the table of a single-GPU run (their digests add up to its digest).
 * When a shared-memory unit overflows on any GPU (one k-mer with more instances than a unit holds, e.g. homopolymer-rich reads), every
 * GPU redoes its shard in instance-record form (gbin_scan_reads_device, gbin_partition_records_device, a gather of every GPU's part
 * by its owner, gbin_group_records_device): same result.  It refuses every descriptor gbin_bin_reads_host refuses, with the same
 * codes, before any GPU starts. */
typedef struct gbin_multi gbin_multi;
int gbin_multi_create(const gbin_config *cfg, const int *devices, int n_devices, gbin_multi **out);
void gbin_multi_destroy(gbin_multi *m);
int gbin_multi_devices(const gbin_multi *m);
gbin_ctx *gbin_multi_context(gbin_multi *m, int i);
const char *gbin_multi_last_error(const gbin_multi *m);
int gbin_multi_bin_reads_host(gbin_multi *m, const gbin_reads *reads, gbin_table *tables_out);

/* ---- read sets larger than one device: the table in P owner parts, one part per call ----
 * Part p of P is the table restricted to the m-mer buckets with gbin_owner_of(mmer_code, P) == p: the same table GPU p owns in a
 * P-GPU run; n_instances / n_distinct count that part only.  Digests of the P parts add up to the digest of the whole table.
 * Every call streams ALL reads through the device in chunks (gbin_set_tuning "part_chunk_kb"), keeps the super-k-mer records of
 * part p and groups them, so device memory holds two read chunks + about 1/P of the records and of the table, whatever n_reads is.
 * Arrival index = read index over the whole `reads` (ids as in gbin_bin_reads_host: read_ids[i] or id_base + i); n_reads < 2^32.
 * The host form writes into the context's pinned arena (ctx_owned = 1, valid until the next call), as gbin_bin_reads_host does:
 * digest, dump or gbin_table_clone each part before asking for the next.  n_parts must be 1..65536 and part < n_parts
 * (else GBIN_E_INVALID_ARG).  A part that overflows pipeline 2's units, reads too long for the super-k-mer scan, or a context set
 * to pipeline 1 make the part go through instance records (pipeline 1); gbin_get_pipeline_info reports what made this part. */
int gbin_bin_reads_host_part(gbin_ctx *ctx, const gbin_reads *reads, uint32_t part, uint32_t n_parts, gbin_table *out);
/* Same with reads in DEVICE memory (e.g. from gbin_split_reads_device); the table stays on the device (ctx_owned, on_device = 1). */
int gbin_bin_reads_device_part(gbin_ctx *ctx, const gbin_reads *reads, uint32_t part, uint32_t n_parts, void *stream, gbin_table *out);
/* Smallest P for which one part of a batch of n_instances k-mer instances fits the device's free memory now (model and measured
 * constants: DESIGN.md §5).  GBIN_E_NOMEM when not even 65536 parts fit. */
int gbin_plan_parts(gbin_ctx *ctx, uint64_t n_instances, uint32_t *n_parts_out);

/* ---- main's read loop on the device (binning.c:1154-1166; SURVEY.md 8 row f2) ----
 * Splits a file image in DEVICE memory into reads exactly as `while (fgets(read, read_length_define, file)) { read[--len] = 0; ... }`
 * does: at most read_length_define-1 bytes per read, stopping after a newline, last byte dropped, one read (and id) per fgets
 * return.  *out receives the ragged form with device pointers (data = d_data; starts/lens owned by the context, valid until
 * the next split) ready for gbin_bin_reads_device.  Same result as gbin_read_file_fgets on the host. */
int gbin_split_reads_device(gbin_ctx *ctx, const char *d_data, uint64_t data_bytes, int read_length_define, void *stream, gbin_reads *out);
/* Plain device -> host copy of context-owned device arrays (device tables, the split's starts / lens). */
int gbin_copy_to_host(gbin_ctx *ctx, void *host_dst, const void *device_src, uint64_t bytes);
/* File -> table in one call: read the file into pinned memory, copy it to the device, split it there, run the hot path, copy
 * the table to the context's pinned arena (ctx_owned = 1).  What `main` does up to and including prune_data. */
int gbin_bin_file_host(gbin_ctx *ctx, const char *path, int read_length_define, gbin_table *out);

/* ---- host helpers ---- */

/* main's read loop (binning.c:1154-1166) over a file: fgets(buf, read_length_define), drop the last
 * char, one read id per fgets return.  Outputs are malloc'ed (free with free()). */
int gbin_read_file_fgets(const char *path, int read_length_define, char **data_out, uint64_t *data_bytes_out,
                         uint64_t **starts_out, uint32_t **lens_out, uint64_t *n_reads_out);
/* Writes "<mmer> <kmer> <id> <id> ...\n" per surviving k-mer of a HOST table to `path` ("-" = stdout). */
int gbin_table_dump(const gbin_table *host, const char *path);
/* Writes the table in print_kmer_read_ids's layout *before* expand_read_id_list (binning.c:792-823):
 * m-mer line, then per k-mer a key line and one line of ids, blank line after each bucket. */
int gbin_table_dump_reference_format(const gbin_table *host, const char *path);
/* Same after expand_read_id_list (binning.c:857-888): every base of a surviving k-mer carries its own copy of the id list,
 * so print_kmer_read_ids prints K lines of ids per k-mer — the layout generate_reads.py:14-62 parses. */
int gbin_table_dump_expanded_format(const gbin_table *host, const char *path);

/* ---- expand_read_id_list (binning.c:857-888): every base of every surviving k-mer gets its own copy of the k-mer's id list ----
 * CSR again: list (j, b) of k-mer j (table order) and base b is ids[list_off[j*K + b] .. list_off[j*K + b + 1]); the K lists of a
 * k-mer are stored back to back.  n_lists = n_kmers * K, n_ids = K * (the table's n_ids): K times the memory of the table's ids. */
typedef struct gbin_expanded {
    int32_t kmer_size;
    int32_t on_device;   /* 1: device pointers owned by the context (valid until its next gbin_expand_read_ids_device call) */
    uint64_t n_lists, n_ids;
    uint64_t *list_off;  /* [n_lists + 1] */
    int32_t *ids;        /* [n_ids] */
} gbin_expanded;
/* Device table in, expanded lists out (device memory of the context).  GBIN_E_TOO_LARGE when K * n_ids ids do not fit the device. */
int gbin_expand_read_ids_device(gbin_ctx *ctx, const gbin_table *dev_table, void *stream, gbin_expanded *out);
/* Copies a device result into malloc'ed host arrays (release with gbin_expanded_free). */
int gbin_expanded_to_host(gbin_ctx *ctx, const gbin_expanded *dev, gbin_expanded *host);
void gbin_expanded_free(gbin_expanded *host);
/* gbin_table_dump_expanded_format's text, written from the expanded lists themselves (what print_kmer_read_ids, binning.c:792-823,
 * prints when it walks the list of lists).  `table` and `lists` are HOST objects of the same batch. */
int gbin_table_dump_expanded_lists(const gbin_table *table, const gbin_expanded *lists, const char *path);

/* ---- the reference's own entry points (binning.c) ---- */
struct ZHashTable;
int getval(char c);            /* binning.c:91 */
char getbp(int bp);            /* binning.c:69 */
int getscore(char *string);    /* binning.c:114 */
/* Enqueues the read (copied; the caller's buffer is not retained) for the table; work happens at
 * prune_data.  Returns hash_table, as the reference does (binning.c:1075). */
struct ZHashTable *process_read(struct ZHashTable *hash_table, char *read, int read_id);
/* Flush point: runs the GPU pipeline over everything enqueued for hash_table and materialises the
 * pruned two-level table into *hash_table using the reference's struct layouts, so unmodified
 * downstream reference code (iterate_level_one_hash, zhash_get, print_kmers ...) can consume it.
 * Returns hash_table (the reference falls off the end without returning, binning.c:1130-1144). */
struct ZHashTable *prune_data(struct ZHashTable *hash_table);
/* K / M / cutoff / device used by process_read + prune_data (defaults 31 / 4 / 1 / 0 = binning.c:10-12). */
int gbin_ref_configure(int kmer_size, int mmer_size, int abundance_cutoff, int device);
/* Status of the last process_read / prune_data call (they cannot return one). */
int gbin_ref_last_status(void);
/* Forgets the staging session bound to a table pointer (so the address can be reused for a new table). */
void gbin_ref_reset(struct ZHashTable *hash_table);
/* Builds the reference pointer graph for a HOST table into *into (an empty table from
 * zcreate_hash_table, or zeroed memory). Keys are strcpy-owned by the table (zhash.c:148-161). */
int gbin_table_to_zhash(const gbin_table *host, struct ZHashTable *into);
/* Frees a graph built by gbin_table_to_zhash / prune_data (entries, keys, lists; not the root struct). */
void gbin_zhash_release(struct ZHashTable *table);

#ifdef __cplusplus
}
#endif
#endif
