// skr_group.cu — pipeline v2: level-2 grouping, prune and emit, in shared memory.
//
// Input: super-k-mer records (skr.cuh) stably sorted by m-mer code, i.e. level 1 of the reference's
// two-level store (binning.c:1044-1049) is already formed and, inside a bucket, records are in arrival
// order.  This file
//   1. plans *units*: runs of whole m-mer buckets whose k-mer instances fit one CTA's shared memory
//      (small buckets packed by windows of T instances; a bucket larger than CAP is expanded ONCE into
//      (k-mer, arrival) records in HBM, range-partitioned on the 64-bit prefix of the oriented k-mer:
//      fine splitters come from a sorted sample of the bucket, exact fine counts are taken, and
//      adjacent fine ranges are merged greedily into slices that fill a unit — ascending k-mer order
//      is kept across the slices);
//   2. runs a persistent kernel, one unit at a time per CTA, that expands the windows of every
//      record (rolling 2-bit shift, complement when is_rev — binning.c:1029-1040), groups equal
//      (m-mer, k-mer) keys with a shared-memory hash (level-2 zhash insert + ll_node push,
//      binning.c:1052-1069), applies the prune (count > ABUNDANCE_CUTOFF, binning.c:1094-1102),
//      sorts the survivors by key, orders every id list newest-first and writes the flat table at
//      offsets obtained from a chained scan over units (so the output is in canonical order);
//   3. derives the bucket directory (mmer_codes / mmer_kmer_off) from the emitted k-mers
//      (prune_data drops buckets that lost all their k-mers, binning.c:1136-1142).
// Anything that does not fit (a single key with more instances than a unit can hold, skewed
// sub-units) raises an overflow flag; the caller then runs the batch through pipeline v1.
#include "gbin_ctx.h"
#include "gbin_device.cuh"
#include "prefix_scan.cuh"
#include "lookback.cuh"
#include "skr.cuh"

namespace gbin {

// A unit holds at most CAP = G_UNIT_CAP k-mer instances (1280: four CTAs per SM).
//   small buckets (<= t = CAP/2 instances) are packed into windows of win = CAP/2 instances of the small-bucket
//   prefix space, so a packed unit holds less than win + t = CAP instances and is about half full on average;
//   a bucket with t < c <= CAP is a unit of its own; a larger one is cut into slices of about tsub = CAP/2.
constexpr uint32_t G_UNIT_CAP = 1280;
struct PlanParams {
    uint32_t cap, t, win, tsub;
};
constexpr int G_RANK_MAX = 512;  // up to this many survivors per unit are ordered by counting instead of a bitonic sort
                                 // (their keys, 20 B each for 128-bit codes, plus a u16 rank array must fit the dead hash table: 16 KB at CAP 1280)

struct __align__(16) Unit {
    uint32_t skr_begin, skr_end;  // range of sorted super-k-mer records; UNIT_RECORDS: range of expanded instance records
    uint32_t flags;               // UNIT_RECORDS: a slice of a bucket larger than CAP, already expanded into the scratch arrays
    uint32_t base_pref;           // instance prefix of the unit's first k-mer instance (its coordinate in the staging arrays)
    uint32_t n_cand;              // k-mer instances of the unit
    uint32_t mmer;                // UNIT_RECORDS: the bucket's m-mer code
    uint32_t pad[2];
};
constexpr uint32_t UNIT_RECORDS = 1u;

// ------------------------------------------------------------------ planning

// Planning reads the 8-byte side records the last sort pass wrote ({m-mer code << 32 | windows}, sorted order), not the records.
struct SkrCount {  // windows of record i
    const uint64_t *side;
    __device__ __forceinline__ uint32_t operator()(uint64_t i) const { return (uint32_t)side[i] & 0xffu; }
};
struct SkrRunHead {
    const uint64_t *side;
    __device__ __forceinline__ uint32_t operator()(uint64_t i) const { return (i == 0 || (side[i] >> 32) != (side[i - 1] >> 32)) ? 1u : 0u; }
};

struct SkrCountAndHead {  // low half: windows of record i; high half: 1 if record i starts a new m-mer run
    const uint64_t *side;
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const {
        return (uint64_t)SkrCount{side}(i) | ((uint64_t)SkrRunHead{side}(i) << 32);
    }
};

// both[i] = exclusive {windows, run heads} before record i (packed u64).  Splits it into inst_prefix[] and run_start[].
__global__ void skr_run_starts_kernel(const uint64_t *__restrict__ side, uint64_t n, const uint64_t *__restrict__ both,
                                      const uint64_t *__restrict__ total, uint32_t *__restrict__ inst_prefix, uint32_t *__restrict__ run_start,
                                      uint32_t *__restrict__ n_inst_out, uint32_t *__restrict__ n_runs_out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t b = both[i];
    inst_prefix[i] = (uint32_t)b;
    if (SkrRunHead{side}(i)) run_start[b >> 32] = (uint32_t)i;
    if (i == n - 1) {
        const uint64_t t = *total;
        inst_prefix[n] = (uint32_t)t;
        run_start[t >> 32] = (uint32_t)n;
        *n_inst_out = (uint32_t)t;
        *n_runs_out = (uint32_t)(t >> 32);
    }
}

struct RunView {
    const uint32_t *run_start;    // [NR+1]
    const uint32_t *inst_prefix;  // [n_skr+1]
    __device__ __forceinline__ uint32_t size(uint64_t r) const { return inst_prefix[run_start[r + 1]] - inst_prefix[run_start[r]]; }
};
struct SmallSize {  // instances of run r if it is a small run, else 0
    RunView rv;
    PlanParams pp;
    __device__ __forceinline__ uint32_t operator()(uint64_t r) const {
        const uint32_t c = rv.size(r);
        return c <= pp.t ? c : 0u;
    }
};
__device__ __forceinline__ uint32_t units_of_big(uint32_t c, const PlanParams &pp) {
    return c > pp.cap ? (c + pp.tsub - 1) / pp.tsub : 1u;  // slices of a bucket that does not fit one unit
}
struct UnitsOfRun {  // how many units start at run r
    RunView rv;
    const uint32_t *small_prefix;  // exclusive sum of SmallSize
    PlanParams pp;
    __device__ __forceinline__ uint32_t operator()(uint64_t r) const {
        const uint32_t c = rv.size(r);
        if (c > pp.t) return units_of_big(c, pp);
        if (r == 0) return 1u;
        if (rv.size(r - 1) > pp.t) return 1u;  // a big bucket closes the packing window
        return (small_prefix[r] / pp.win != small_prefix[r - 1] / pp.win) ? 1u : 0u;
    }
};

__device__ __forceinline__ unsigned int *big_counter(GroupCounters *gc);
__device__ __forceinline__ unsigned int *big_inst_counter(GroupCounters *gc);

__global__ void fill_units_kernel(RunView rv, const uint32_t *__restrict__ small_prefix, const uint32_t *__restrict__ unit_base,
                                  uint64_t n_runs, PlanParams pp, Unit *__restrict__ units, GroupCounters *__restrict__ gc,
                                  uint32_t *__restrict__ big_list) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint32_t nu = UnitsOfRun{rv, small_prefix, pp}(r);
    const uint32_t c = rv.size(r);
    const uint32_t ub = unit_base[r];
    if (c > pp.cap) {
        // sliced bucket: partition_big_runs_kernel expands it into the scratch arrays and fills its units
        const uint32_t bi = atomicAdd(big_counter(gc), 1u);
        big_list[2 * bi] = (uint32_t)r;
        big_list[2 * bi + 1] = atomicAdd(big_inst_counter(gc), c);  // its base in the scratch arrays
    } else if (c > pp.t) {
        units[ub] = Unit{rv.run_start[r], rv.run_start[r + 1], 0u, rv.inst_prefix[rv.run_start[r]], c, 0u, {0u, 0u}};
    } else {
        // unit of this run = the latest head at or before it: exclusive base + own head flag - 1
        const uint32_t u = ub + nu - 1;
        if (nu) {
            units[u].skr_begin = rv.run_start[r];
            units[u].flags = 0;
            units[u].base_pref = rv.inst_prefix[rv.run_start[r]];
        }
        atomicMax(&units[u].skr_end, rv.run_start[r + 1]);
        atomicAdd(&units[u].n_cand, c);
    }
}

// Calls f(t, k0, k1, prefix) for the windows t = t0, t0 + step, ... of a super-k-mer record: the oriented k-mer code (top 2K bits
// of the payload shifted left by t bases, complemented when is_rev — binning.c:1029-1040) and its 64-bit prefix (monotone in the
// code).  step * 2 < 64.  (t0, step) = (0, 1) walks every window; the grouping kernel shares a record among several threads.
template <int PW, int KW, typename F>
__device__ __forceinline__ void for_each_window_strided(const uint32_t *__restrict__ rec, int K, uint32_t t0, uint32_t step, F &&f) {
    const uint4 *p = reinterpret_cast<const uint4 *>(rec);
    const uint4 h = p[0];
    const uint32_t n = h.z & 0xffu;
    const bool rev = (h.z >> 8) & 1u;
    const uint64_t kmask0 = (2 * K >= 64 * KW) ? ~0ull : ((1ull << (2 * K - 64 * (KW - 1))) - 1);  // mask of the most significant word
    uint64_t w[PW];
    {
        const uint4 a = p[1];
        w[0] = ((uint64_t)a.x << 32) | a.y;
        w[1] = ((uint64_t)a.z << 32) | a.w;
        if (PW == 4) {
            const uint4 b = p[2];
            w[PW - 2] = ((uint64_t)b.x << 32) | b.y;
            w[PW - 1] = ((uint64_t)b.z << 32) | b.w;
        }
    }
    auto advance = [&](uint32_t bases) {  // 0 < 2 * bases < 64
        const uint32_t sh = 2 * bases;
#pragma unroll
        for (int q = 0; q < PW - 1; q++) w[q] = (w[q] << sh) | (w[q + 1] >> (64 - sh));
        w[PW - 1] <<= sh;
    };
    if (t0) advance(t0);
    for (uint32_t t = t0; t < n; t += step) {
        uint64_t k0, k1 = 0;
        if (KW == 1) {
            k0 = (2 * K == 64) ? w[0] : (w[0] >> (64 - 2 * K));
            if (rev) k0 = ~k0 & kmask0;
        } else {
            const int r = 128 - 2 * K;  // 0..62
            k0 = r ? (w[0] >> r) : w[0];
            k1 = r ? ((w[1] >> r) | (w[0] << (64 - r))) : w[1];
            if (rev) {
                k0 = ~k0 & kmask0;
                k1 = ~k1;
            }
        }
        uint64_t pre = rev ? ~w[0] : w[0];
        if (2 * K < 64) pre &= ~0ull << (64 - 2 * K);
        f(t, k0, k1, pre);
        advance(step);
    }
}
template <int PW, int KW, typename F>
__device__ __forceinline__ void for_each_window(const uint32_t *__restrict__ rec, int K, F &&f) {
    for_each_window_strided<PW, KW>(rec, K, 0u, 1u, f);
}

// 64-bit prefix of the oriented k-mer of window w of a record (random access form of the above).
template <int PW>
__device__ __forceinline__ uint64_t window_prefix(const uint32_t *rec, uint32_t w, int K) {
    const uint32_t bit = 2 * w, wi = bit >> 5, sh = bit & 31;
    const uint32_t *pl = rec + 4;
    auto word = [&](uint32_t i) -> uint32_t { return i < 2u * PW ? pl[i] : 0u; };
    const uint32_t a = __funnelshift_l(word(wi + 1), word(wi), sh);
    const uint32_t b = __funnelshift_l(word(wi + 2), word(wi + 1), sh);
    uint64_t pre = ((uint64_t)a << 32) | b;
    if ((rec[2] >> 8) & 1u) pre = ~pre;
    if (2 * K < 64) pre &= ~0ull << (64 - 2 * K);
    return pre;
}

constexpr int PART_THREADS = 256;
constexpr int PART_SAMPLES = 2048;  // sorted sample of k-mer prefixes of one bucket
constexpr int PART_FINE = 1024;     // fine ranges the bucket is counted into before they are merged into slices
                                    // (32 KB of shared memory in total, so several buckets are in flight per SM)

struct BigScratch {
    uint64_t *k0, *k1;  // k-mer code words of the expanded instances (k1 only for 128-bit codes)
    uint32_t *arr;      // their arrival indices
};

// One CTA per bucket larger than a unit.  (1) Sample the bucket's k-mer prefixes evenly over its instances and sort the
// sample.  (2) Take fine splitters from it (fine ranges of about CAP/8 instances), expand every window once and count the
// fine ranges exactly.  (3) Merge adjacent fine ranges greedily into slices of at most CAP instances — these are the
// bucket's units, in ascending k-mer order.  (4) Expand again and scatter (k-mer, arrival) to the slice-major scratch.
template <int PW, int KW>
__global__ void __launch_bounds__(PART_THREADS)
    partition_big_runs_kernel(const uint32_t *__restrict__ skr, RunView rv, const uint32_t *__restrict__ unit_base,
                              const uint32_t *__restrict__ big_list, GroupCounters *__restrict__ gc, PlanParams pp, int K, BigScratch sc,
                              Unit *__restrict__ units) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    extern __shared__ __align__(16) uint8_t part_smem[];
    uint64_t *samp = reinterpret_cast<uint64_t *>(part_smem);         // [PART_SAMPLES]
    uint64_t *spl = samp + PART_SAMPLES;                              // [PART_FINE] fine splitters (spl[0] unused)
    uint32_t *cnt = reinterpret_cast<uint32_t *>(spl + PART_FINE);    // [PART_FINE] fine counts, then scatter cursors
    uint32_t *foff = cnt + PART_FINE;                                 // [PART_FINE + 1] exclusive prefix of the fine counts
    __shared__ uint32_t s_bad;
    __shared__ uint16_t lut[258];  // lut[b] = fine range of the smallest prefix whose top byte is b
    const uint32_t nb = gc->n_big;
    for (uint32_t bi = blockIdx.x; bi < nb; bi += gridDim.x) {
        const uint64_t r = big_list[2 * bi];
        const uint32_t sbase = big_list[2 * bi + 1];
        const uint32_t c = rv.size(r);
        const uint32_t a = rv.run_start[r], b = rv.run_start[r + 1];
        const uint32_t base = rv.inst_prefix[a];
        const uint32_t P = units_of_big(c, pp);  // unit slots reserved for this bucket
        const uint32_t mmer = skr[(uint64_t)a * NW + 1];
        uint32_t F = (c + pp.cap / 8 - 1) / (pp.cap / 8);  // fine ranges
        if (F > (uint32_t)PART_FINE) F = PART_FINE;
        uint32_t S = 128;  // samples: a power of two, about 8 per fine range, at most PART_SAMPLES
        while (S < 8 * F && S < (uint32_t)PART_SAMPLES) S <<= 1;
        if (threadIdx.x == 0) s_bad = 0;
        // ---- (1) sample + sort
        for (uint32_t t = threadIdx.x; t < S; t += PART_THREADS) {
            const uint32_t j = (uint32_t)(((uint64_t)(2 * t + 1) * c) / (2ull * S));  // instance index inside the bucket
            uint32_t lo = a, hi = b - 1;  // last record whose first instance is <= j
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (rv.inst_prefix[mid] - base <= j) lo = mid;
                else hi = mid - 1;
            }
            samp[t] = window_prefix<PW>(skr + (uint64_t)lo * NW, j - (rv.inst_prefix[lo] - base), K);
        }
        __syncthreads();
        for (uint32_t k = 2; k <= S; k <<= 1) {
            for (uint32_t jj = k >> 1; jj > 0; jj >>= 1) {
                for (uint32_t idx = threadIdx.x; idx < S; idx += PART_THREADS) {
                    const uint32_t partner = idx ^ jj;
                    if (partner > idx) {
                        const uint64_t x = samp[idx], y = samp[partner];
                        if ((x > y) == ((idx & k) == 0)) {
                            samp[idx] = y;
                            samp[partner] = x;
                        }
                    }
                }
                __syncthreads();
            }
        }
        // ---- (2) fine splitters and exact fine counts.  fine range f holds prefixes in [spl[f], spl[f+1])
        for (uint32_t f = threadIdx.x; f < F; f += PART_THREADS) {
            spl[f] = f ? samp[(uint64_t)f * S / F] : 0ull;
            cnt[f] = 0;
        }
        __syncthreads();
        auto fine_search = [&](uint64_t pre) -> uint32_t {  // number of splitters spl[1..F-1] that are <= pre
            uint32_t lo = 0, hi = F - 1;
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (spl[mid] <= pre) lo = mid;
                else hi = mid - 1;
            }
            return lo;
        };
        // a 256-entry table on the top byte of the prefix narrows the search to a step or two
        for (uint32_t bb = threadIdx.x; bb < 257; bb += PART_THREADS) lut[bb] = bb < 256 ? (uint16_t)fine_search((uint64_t)bb << 56) : (uint16_t)(F - 1);
        __syncthreads();
        // the k-mers of a bucket share long prefixes (every window whose signature sits at offset j starts with j free bases
        // followed by the m-mer itself), so the top byte alone leaves long candidate ranges: bisect inside the table's range
        auto fine_of = [&](uint64_t pre) -> uint32_t {
            const uint32_t bb = (uint32_t)(pre >> 56);
            uint32_t lo = lut[bb], hi = lut[bb + 1];  // the answer is the last f in [lo, hi] with spl[f] <= pre (spl[lo] <= pre holds)
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (spl[mid] <= pre) lo = mid;
                else hi = mid - 1;
            }
            return lo;
        };
        for (uint32_t s = a + threadIdx.x; s < b; s += PART_THREADS)
            for_each_window<PW, KW>(skr + (uint64_t)s * NW, K, [&](uint32_t, uint64_t, uint64_t, uint64_t pre) { atomicAdd(&cnt[fine_of(pre)], 1u); });
        __syncthreads();
        // ---- (3) greedy merge of adjacent fine ranges into slices of at most CAP instances (one thread: F is small)
        if (threadIdx.x == 0) {
            const uint32_t ub = unit_base[r];
            uint32_t q = 0, run = 0, start = 0, acc = 0;
            for (uint32_t f = 0; f < F; f++) {
                const uint32_t cf = cnt[f];
                foff[f] = acc;
                if (cf > pp.cap) s_bad = 1;  // one fine range (one k-mer prefix, typically one k-mer) overflows a unit
                if (run + cf > pp.cap) {
                    if (q < P) units[ub + q] = Unit{sbase + start, sbase + acc, UNIT_RECORDS, base + start, run, mmer, {0u, 0u}};
                    q++;
                    start = acc;
                    run = 0;
                }
                run += cf;
                acc += cf;
            }
            foff[F] = acc;
            if (q < P) units[ub + q] = Unit{sbase + start, sbase + acc, UNIT_RECORDS, base + start, run, mmer, {0u, 0u}};
            q++;
            if (q > P || acc != c) s_bad = 1;
            for (; q < P; q++) units[ub + q] = Unit{sbase + acc, sbase + acc, UNIT_RECORDS, base + acc, 0u, mmer, {0u, 0u}};  // unused slots: empty units
        }
        __syncthreads();
        if (s_bad) {
            if (threadIdx.x == 0) atomicExch(&gc->overflow, 4u);
            __syncthreads();
            continue;
        }
        for (uint32_t f = threadIdx.x; f < F; f += PART_THREADS) cnt[f] = 0;
        __syncthreads();
        // ---- (4) expand again and scatter to the slice-major scratch (order inside a fine range is arbitrary)
        for (uint32_t s = a + threadIdx.x; s < b; s += PART_THREADS) {
            const uint32_t *rec = skr + (uint64_t)s * NW;
            const uint32_t arrival = rec[0];
            for_each_window<PW, KW>(rec, K, [&](uint32_t, uint64_t k0, uint64_t k1, uint64_t pre) {
                const uint32_t f = fine_of(pre);
                const uint64_t pos = (uint64_t)sbase + foff[f] + atomicAdd(&cnt[f], 1u);
                sc.k0[pos] = k0;
                if (KW == 2) sc.k1[pos] = k1;
                sc.arr[pos] = arrival;
            });
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ grouping kernel

// Named barriers of the grouping kernel: 0 = the whole CTA (workers + control warp), 1 = the workers only,
// 2 = "the unit's totals are published" (workers arrive, the control warp waits).
__device__ __forceinline__ void bar_workers(int n) { asm volatile("bar.sync 1, %0;" ::"r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_wait(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_all() { asm volatile("bar.sync 0;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Exclusive scan over the NT worker threads (barrier 1).
template <int NT>
__device__ __forceinline__ uint32_t block_excl_scan_u32(uint32_t v, uint32_t *total, uint32_t *warp_sums /* NT/32 + 1 */) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (unsigned)d) inc += o;
    }
    if (lane == 31) warp_sums[warp] = inc;
    bar_workers(NT);
    if (warp == 0) {
        uint32_t s = lane < NT / 32 ? warp_sums[lane] : 0u;
        uint32_t si = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, si, d);
            if (lane >= (unsigned)d) si += o;
        }
        if (lane < NT / 32) warp_sums[lane] = si - s;
        if (lane == NT / 32 - 1) warp_sums[NT / 32] = si;
    }
    bar_workers(NT);
    const uint32_t res = inc - v + warp_sums[warp];
    *total = warp_sums[NT / 32];
    bar_workers(NT);
    return res;
}

struct GroupOut {
    uint64_t *kmer_codes;   // [S*KW]
    uint32_t *kmer_mmer;    // [S]
    uint64_t *kmer_id_off;  // [S+1]
    int32_t *read_ids;      // [N]
    uint64_t kmer_cap, id_cap;
    // staging: a unit writes its part of the table at a place that depends on the unit alone (instance coordinate for ids,
    // instance coordinate / (cutoff + 1) for k-mers), and the CTA moves it to its final place one unit later, when the
    // chained scan over units has long resolved — nobody ever waits for a predecessor
    int32_t *stg_ids;       // [id_cap]
    uint64_t *stg_codes;    // [kmer_cap * KW]
    uint32_t *stg_mmer;     // [kmer_cap]
    uint32_t *stg_off;      // [kmer_cap] start of the k-mer's id list inside its unit
};

__device__ __forceinline__ unsigned int *big_counter(GroupCounters *gc) { return &gc->n_big; }
__device__ __forceinline__ unsigned int *big_inst_counter(GroupCounters *gc) { return &gc->big_inst; }

template <int KW>
__device__ __forceinline__ bool key_less(const uint64_t *key0, const uint64_t *key1, const uint32_t *mm, uint32_t a, uint32_t b) {
    if (mm[a] != mm[b]) return mm[a] < mm[b];
    if (key0[a] != key0[b]) return key0[a] < key0[b];
    if (KW == 2) return key1[a] < key1[b];
    return false;
}

// The CTA = G_THREADS worker threads + one control warp.  The workers run the phases of a unit separated by barrier 1;
// the control warp hides the latencies that are serial per unit: it resolves the unit's output offsets (chained scan over
// units) while the workers order the survivors, and it takes the next ticket, fetches the next unit's descriptor and
// prefetches its records into L2 while the workers write the unit's output.
template <int PW, int KW, int G_CAP, int G_THREADS>
__global__ void __launch_bounds__(G_THREADS + 32)
    skr_group_kernel(const uint32_t *__restrict__ skr, const uint32_t *__restrict__ inst_prefix, const Unit *__restrict__ units, BigScratch sc,
                     int K, int cutoff, const int32_t *__restrict__ ids_by_arrival, int32_t id_base, GroupOut out,
                     unsigned long long *__restrict__ unit_state, GroupCounters *__restrict__ gc, uint32_t chunk, uint32_t n_chunks,
                     uint32_t *__restrict__ chunk_tickets) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    constexpr int ALL = G_THREADS + 32;
    constexpr int G_LOG_HS = G_CAP > 2048 ? 13 : (G_CAP > 1024 ? 12 : 11);
    constexpr int G_HS = 1 << G_LOG_HS;  // hash slots: the power of two in [2 CAP, 4 CAP)
    static_assert(G_CAP % G_THREADS == 0 && G_CAP > 1024 && G_CAP <= 4096, "unit capacity");
    static_assert((size_t)G_RANK_MAX * (8 * KW + 4 + 2) <= (size_t)G_HS * 4, "the survivors' keys and ranks are laid over the dead hash table");
    extern __shared__ __align__(16) uint8_t smem[];
    uint64_t *key0 = reinterpret_cast<uint64_t *>(smem);
    uint64_t *key1 = key0 + (KW == 2 ? G_CAP : 0);
    uint32_t *mm = reinterpret_cast<uint32_t *>(key0 + KW * G_CAP);
    uint32_t *arr = mm + G_CAP;
    uint32_t *table = arr + G_CAP;  // G_HS slots; after grouping: [0,CAP) id offsets of survivors, [CAP,2*CAP) scratch / staged ids
    uint32_t *cnt = table + G_HS;
    uint16_t *grp = reinterpret_cast<uint16_t *>(cnt + G_CAP);
    uint16_t *rnk = grp + G_CAP;
    uint16_t *surv = rnk + G_CAP;
    uint32_t *off = table;                 // off[s], s < S <= CAP (the end of the last list is the unit's id total)
    uint32_t *stage_ids = table + G_CAP;   // scratch; together with cnt (free once the offsets exist) 2*CAP words
    __shared__ uint32_t s_nsurv, s_ndistinct, s_scan[G_THREADS / 32 + 1];
    __shared__ unsigned long long s_agg;
    __shared__ uint32_t s_total_ids;
    __shared__ uint32_t s_uidx[2];
    __shared__ Unit s_un[2];

    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const bool ctrl = tid >= (uint32_t)G_THREADS;

    // One launch handles chunk `chunk` of `n_chunks` equal ranges of the unit list (the host path streams the finished part
    // of the table to the host while later chunks are still being grouped); the chained scan runs across the launches.
    const uint32_t n_units_all = gc->n_units;
    const uint32_t unit_begin = (uint32_t)(((uint64_t)n_units_all * chunk) / n_chunks);
    const uint32_t n_units = (uint32_t)(((uint64_t)n_units_all * (chunk + 1)) / n_chunks);  // this launch handles [unit_begin, n_units)
    uint32_t *chunk_ticket = chunk_tickets + chunk;

    // Control warp: units are handed out by an atomic ticket, taken while the CTA orders and stages its current unit — a ticket
    // taken much earlier would let later units overtake it, and their chained-scan resolve would then wait for it.
    auto fetch_unit = [&](int slot) {
        uint32_t u = 0;
        if (lane == 0) u = unit_begin + atomicAdd(chunk_ticket, 1u);
        u = __shfl_sync(0xffffffffu, u, 0);
        if (lane == 0) s_uidx[slot] = u;
        if (u >= n_units) return;
        const uint32_t w = lane < 8 ? reinterpret_cast<const uint32_t *>(units + u)[lane] : 0u;
        if (lane < 8) reinterpret_cast<uint32_t *>(&s_un[slot])[lane] = w;
        const uint32_t b = __shfl_sync(0xffffffffu, w, 0), e = __shfl_sync(0xffffffffu, w, 1), fl = __shfl_sync(0xffffffffu, w, 2);
        if (fl & UNIT_RECORDS) {
            const char *p0 = reinterpret_cast<const char *>(sc.k0 + b), *p1 = reinterpret_cast<const char *>(sc.k0 + e);
            for (const char *p = p0 + 128 * lane; p < p1; p += 128 * 32) prefetch_l2(p);
            const char *q0 = reinterpret_cast<const char *>(sc.arr + b), *q1 = reinterpret_cast<const char *>(sc.arr + e);
            for (const char *p = q0 + 128 * lane; p < q1; p += 128 * 32) prefetch_l2(p);
            if (KW == 2) {
                const char *r0 = reinterpret_cast<const char *>(sc.k1 + b), *r1 = reinterpret_cast<const char *>(sc.k1 + e);
                for (const char *p = r0 + 128 * lane; p < r1; p += 128 * 32) prefetch_l2(p);
            }
        } else {
            const char *p0 = reinterpret_cast<const char *>(skr + (uint64_t)b * NW), *p1 = reinterpret_cast<const char *>(skr + (uint64_t)e * NW);
            for (const char *p = p0 + 128 * lane; p < p1; p += 128 * 32) prefetch_l2(p);
            const char *q0 = reinterpret_cast<const char *>(inst_prefix + b), *q1 = reinterpret_cast<const char *>(inst_prefix + e);
            for (const char *p = q0 + 128 * lane; p < q1; p += 128 * 32) prefetch_l2(p);
        }
    };

    // What the CTA still has to move from the staging arrays to its final place: the unit it finished last.
    bool have_prev = false;
    uint32_t prev_u = 0, prev_S = 0, prev_N = 0, prev_idb = 0, prev_kb = 0;
    const uint32_t kdiv = cutoff >= 0 ? (uint32_t)cutoff + 1u : 1u;  // a surviving k-mer has more than `cutoff` instances

    // Control warp, previous unit: resolve its output offsets from the chained scan over units — one unit late, so its
    // predecessors have published long ago and nobody ever waits for a laggard (resolving at once and letting the workers
    // wait at the end of the unit was measured 1.5x slower on batches with few survivors per unit)
    auto resolve_prev = [&]() -> unsigned long long {
        const unsigned long long agg = ((unsigned long long)prev_S << 31) | prev_N;
        const unsigned long long base = lkb_resolve_warp<8>(unit_state, prev_u, agg, lane);  // the same value in every lane
        if (lane == 0 && prev_u == n_units_all - 1) {
            gc->total_kmers = (base >> 31) + prev_S;
            gc->total_ids = (base & 0x7fffffffull) + prev_N;
        }
        return base;
    };
    // Control warp, previous unit: staging -> final place (the data is still in L2; eight loads in flight per lane)
    auto move_prev = [&](unsigned long long pb) {
        const uint64_t S_base = pb >> 31, N_base = pb & 0x7fffffffull;
        if (S_base + prev_S > out.kmer_cap || N_base + prev_N > out.id_cap) {  // cannot happen with the caller's bounds; never write out of range
            if (lane == 0) atomicExch(&gc->overflow, 2u);
            return;
        }
        const int32_t *src = out.stg_ids + prev_idb;
        int32_t *dst = out.read_ids + N_base;
        uint32_t i = lane;
        for (; i + 7 * 32 < prev_N; i += 8 * 32) {
            int32_t v[8];
#pragma unroll
            for (int k = 0; k < 8; k++) v[k] = __ldcg(src + i + 32 * k);
#pragma unroll
            for (int k = 0; k < 8; k++) dst[i + 32 * k] = v[k];
        }
        for (; i < prev_N; i += 32) dst[i] = __ldcg(src + i);
        for (uint32_t x = lane; x < prev_S; x += 32) {
            const uint64_t g = S_base + x, q = (uint64_t)prev_kb + x;
            out.kmer_codes[g * KW] = __ldcg(out.stg_codes + q * KW);
            if (KW == 2) out.kmer_codes[g * KW + 1] = __ldcg(out.stg_codes + q * KW + 1);
            out.kmer_mmer[g] = __ldcg(out.stg_mmer + q);
            out.kmer_id_off[g] = N_base + __ldcg(out.stg_off + q);
        }
    };

    if (ctrl) fetch_unit(0);
    bar_all();
    for (int cur = 0;; cur ^= 1) {
        const uint32_t u = s_uidx[cur];
        if (u >= n_units) break;
        const Unit un = s_un[cur];
        const uint32_t n_cand = un.n_cand;
        const bool too_big = n_cand > (uint32_t)G_CAP;  // cannot happen with the planner's bounds; the batch is then redone by pipeline v1
        const uint32_t idb = un.base_pref, kb = un.base_pref / kdiv;  // this unit's places in the staging arrays

        if (ctrl) {
            if (have_prev) move_prev(resolve_prev());  // while the workers expand and group this unit
            bar_wait(2, ALL);                          // the workers have published this unit's totals
            const unsigned long long agg = s_agg;
            fetch_unit(cur ^ 1);
            bar_all();  // Y: the unit is staged
            have_prev = true;
            prev_u = u;
            prev_S = (uint32_t)(agg >> 31);
            prev_N = (uint32_t)(agg & 0x7fffffffull);
            prev_idb = idb;
            prev_kb = kb;
            continue;
        }

        // ================================================================ workers
        const uint32_t base_pref = un.base_pref;
        const bool from_records = (un.flags & UNIT_RECORDS) != 0;  // a slice of a big bucket: its instances arrive in arbitrary order
        if (tid == 0) {
            s_nsurv = 0;
            s_ndistinct = 0;
            s_total_ids = 0;
        }
        // ---- zero the hash table and counters (contiguous: table, cnt) while records stream in
        {
            uint4 *z = reinterpret_cast<uint4 *>(table);
            for (uint32_t i = tid; i < (uint32_t)(G_HS + G_CAP) / 4; i += G_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        if (!too_big) {
            if (from_records) {
                // ---- instances of a big bucket's slice were expanded by partition_big_runs_kernel: just load them
                for (uint32_t i = tid; i < n_cand; i += G_THREADS) {
                    const uint64_t g = (uint64_t)un.skr_begin + i;
                    key0[i] = sc.k0[g];
                    if (KW == 2) key1[i] = sc.k1[g];
                    mm[i] = un.mmer;
                    arr[i] = sc.arr[g];
                }
            } else {
                // ---- expansion: EXP_SUB threads share a super-k-mer record (a unit holds far fewer records than the CTA has
                // threads), thread j of them rolling over the windows j, j + EXP_SUB, ...
                constexpr uint32_t EXP_SUB = 4;
                const uint32_t n_rec = un.skr_end - un.skr_begin;
                for (uint32_t e = tid; e < n_rec * EXP_SUB; e += G_THREADS) {
                    const uint32_t s = un.skr_begin + e / EXP_SUB;
                    const uint32_t *rec = skr + (uint64_t)s * NW;
                    const uint32_t arrival = rec[0], mmer = rec[1];
                    const uint32_t pos0 = inst_prefix[s] - base_pref;
                    for_each_window_strided<PW, KW>(rec, K, e % EXP_SUB, EXP_SUB, [&](uint32_t t, uint64_t k0, uint64_t k1, uint64_t) {
                        const uint32_t pos = pos0 + t;
                        key0[pos] = k0;
                        if (KW == 2) key1[pos] = k1;
                        mm[pos] = mmer;
                        arr[pos] = arrival;
                    });
                }
            }
        }
        bar_workers(G_THREADS);
        if (too_big) {  // give up on this unit (the whole batch will be redone by pipeline v1) but keep the chain alive
            if (tid == 0) {
                atomicExch(&gc->overflow, 1u);
                s_agg = 0ull;
                lkb_publish_aggregate(unit_state, u, 0ull);
            }
            __threadfence_block();
            bar_arrive(2, ALL);
            bar_all();  // Y
            have_prev = true;
            prev_u = u;
            prev_S = prev_N = 0;
            prev_idb = idb;
            prev_kb = kb;
            continue;
        }
        const uint32_t n_inst = n_cand;

        // ---- group: claim a slot with the instance index, compare keys through the instance arrays
        for (uint32_t i = tid; i < n_inst; i += G_THREADS) {
            const uint64_t k0 = key0[i], k1 = (KW == 2) ? key1[i] : 0ull;
            const uint32_t m = mm[i];
            uint32_t hx = ((uint32_t)k0 * 0x9E3779B1u) ^ ((uint32_t)(k0 >> 32) * 0x85EBCA77u) ^ (m * 0xC2B2AE3Du);
            if (KW == 2) hx ^= ((uint32_t)k1 * 0x27D4EB2Fu) ^ ((uint32_t)(k1 >> 32) * 0x165667B1u);
            hx *= 0x9E3779B1u;
            uint32_t h = hx >> (32 - G_LOG_HS);
            uint32_t rep;
            for (;;) {
                uint32_t c = table[h];
                if (c == 0) {
                    c = atomicCAS(&table[h], 0u, i + 1);
                    if (c == 0) {
                        rep = i;
                        break;
                    }
                }
                const uint32_t r = c - 1;
                if (key0[r] == k0 && (KW == 1 || key1[r] == k1) && mm[r] == m) {
                    rep = r;
                    break;
                }
                h = (h + 1) & (G_HS - 1);
            }
            grp[i] = (uint16_t)rep;
            rnk[i] = (uint16_t)atomicAdd(&cnt[rep], 1u);
        }
        bar_workers(G_THREADS);

        // ---- leaders and survivors (keep iff count > cutoff, binning.c:1102)
        for (uint32_t i0 = 0; i0 < n_inst; i0 += G_THREADS) {
            const uint32_t i = i0 + tid;
            const bool leader = i < n_inst && grp[i] == i;
            const unsigned lm = __ballot_sync(0xffffffffu, leader);
            if (lane == 0 && lm) atomicAdd(&s_ndistinct, (uint32_t)__popc(lm));
            if (leader && (cutoff < 0 || cnt[i] > (uint32_t)cutoff)) {
                surv[atomicAdd(&s_nsurv, 1u)] = (uint16_t)i;
                atomicAdd(&s_total_ids, cnt[i]);
            }
        }
        bar_workers(G_THREADS);
        const uint32_t S = s_nsurv, N = s_total_ids;
        // the unit's totals are known before any ordering work: publish them now so that successors rarely wait, and let the
        // control warp resolve this unit's output offsets while the survivors are being ordered
        if (tid == 0) {
            s_agg = ((unsigned long long)S << 31) | N;
            lkb_publish_aggregate(unit_state, u, ((unsigned long long)S << 31) | N);
            atomicAdd(&gc->distinct, (unsigned long long)s_ndistinct);
        }
        __threadfence_block();
        bar_arrive(2, ALL);

        // ---- survivors ascending by (m-mer, k-mer).  Usual case (a few hundred survivors): every survivor counts
        // the survivors with a smaller key (keys are distinct, so ranks are a permutation) — no barriers inside;
        // otherwise a bitonic sort of the instance indices, padded with 0xFFFF = +inf.
        if (S <= (uint32_t)G_RANK_MAX) {
            // the hash table is dead from here on: its memory holds the survivors' keys side by side, so the ranking
            // loop reads consecutive broadcast words instead of chasing surv[] -> key arrays
            uint64_t *sk0 = reinterpret_cast<uint64_t *>(table);
            uint64_t *sk1 = sk0 + (KW == 2 ? G_RANK_MAX : 0);
            uint32_t *smm = reinterpret_cast<uint32_t *>(sk0 + KW * G_RANK_MAX);
            uint16_t *tmp = reinterpret_cast<uint16_t *>(smm + G_RANK_MAX);
            for (uint32_t s = tid; s < S; s += G_THREADS) {
                const uint32_t i = surv[s];
                sk0[s] = key0[i];
                if (KW == 2) sk1[s] = key1[i];
                smm[s] = mm[i];
            }
            bar_workers(G_THREADS);
            for (uint32_t s = tid; s < S; s += G_THREADS) {
                const uint64_t k0 = sk0[s], k1 = (KW == 2) ? sk1[s] : 0ull;
                const uint32_t m = smm[s];
                uint32_t rank = 0;
#pragma unroll 4
                for (uint32_t t = 0; t < S; t++) {
                    const uint32_t mj = smm[t];
                    const uint64_t kj = sk0[t];
                    bool less = mj < m || (mj == m && kj < k0);
                    if constexpr (KW == 2) less = less || (mj == m && kj == k0 && sk1[t] < k1);
                    rank += less ? 1u : 0u;
                }
                tmp[rank] = surv[s];
            }
            bar_workers(G_THREADS);
            for (uint32_t s = tid; s < S; s += G_THREADS) surv[s] = tmp[s];
            bar_workers(G_THREADS);
        } else {
            uint32_t n2 = 1;
            while (n2 < S) n2 <<= 1;
            for (uint32_t i = S + tid; i < n2; i += G_THREADS) surv[i] = 0xFFFFu;
            bar_workers(G_THREADS);
            for (uint32_t k = 2; k <= n2; k <<= 1) {
                for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                    for (uint32_t idx = tid; idx < n2; idx += G_THREADS) {
                        const uint32_t partner = idx ^ j;
                        if (partner > idx) {
                            const uint32_t a = surv[idx], b = surv[partner];
                            // a > b ?  (0xFFFF is larger than everything)
                            const bool gt = (a == 0xFFFFu) ? (b != 0xFFFFu) : (b == 0xFFFFu ? false : key_less<KW>(key0, key1, mm, b, a));
                            const bool asc = (idx & k) == 0;
                            if (gt == asc) {
                                surv[idx] = (uint16_t)b;
                                surv[partner] = (uint16_t)a;
                            }
                        }
                    }
                    bar_workers(G_THREADS);
                }
            }
        }

        // ---- id offsets of the survivors (the hash table is dead from here on: its memory holds stage_ids / off)
        {
            uint32_t carry = 0;
            for (uint32_t b0 = 0; b0 < S; b0 += G_THREADS) {
                const uint32_t s = b0 + tid;
                const uint32_t v = s < S ? cnt[surv[s]] : 0u;
                uint32_t tot;
                const uint32_t ex = block_excl_scan_u32<G_THREADS>(v, &tot, s_scan);
                if (s < S) off[s] = carry + ex;
                carry += tot;
            }
        }
        bar_workers(G_THREADS);

        // ---- every instance learns the index s of its surviving list (0xFFFF: pruned)
        {
            uint16_t *mapv = reinterpret_cast<uint16_t *>(stage_ids);  // leader index -> s
            for (uint32_t sI = tid; sI < S; sI += G_THREADS) mapv[surv[sI]] = (uint16_t)sI;
            bar_workers(G_THREADS);
            for (uint32_t i = tid; i < n_inst; i += G_THREADS) {
                const uint32_t rep = grp[i];
                grp[i] = (cutoff < 0 || cnt[rep] > (uint32_t)cutoff) ? mapv[rep] : (uint16_t)0xFFFFu;
            }
            bar_workers(G_THREADS);
        }

        constexpr int ITERS = G_CAP / G_THREADS;   // instances per thread
        // rows of the (list, chunk) matrix below: one u16 per 32-instance chunk of the unit, padded to an odd number of
        // 32-bit words so that the lanes of a warp (same chunk, different lists) fall into different banks
        const uint32_t nch = (n_inst + 31) >> 5;
        const uint32_t row_words = ((nch + 1) >> 1) | 1u, row = 2 * row_words;
        const bool ordered = !from_records && S * row_words <= 2u * G_CAP;
        if (ordered) {
            // ---- id lists, ordered path.  Instance positions of a unit expanded from super-k-mer records follow arrival order, so the place of
            // an instance in its newest-first list is (members of the list in later chunks) + (members at a higher lane of
            // its own chunk): a per-(list, chunk) count matrix filled with warp match, a suffix sum per list, done.
            uint16_t *mat = reinterpret_cast<uint16_t *>(stage_ids);  // [S][row], spills into cnt (dead by now)
            for (uint32_t x = tid; x < S * row_words; x += G_THREADS) reinterpret_cast<uint32_t *>(mat)[x] = 0u;
            bar_workers(G_THREADS);
            uint32_t within[ITERS];
            const uint32_t gt_mask = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
#pragma unroll
            for (int it = 0; it < ITERS; it++) {
                const uint32_t p = it * G_THREADS + tid;
                within[it] = 0;
                if (it * G_THREADS < n_inst) {
                    const uint32_t sI = p < n_inst ? grp[p] : 0xFFFFu;
                    const bool act = sI != 0xFFFFu;
                    const unsigned amask = __ballot_sync(0xffffffffu, act);
                    if (act) {
                        const unsigned peers = __match_any_sync(amask, sI);
                        within[it] = __popc(peers & gt_mask);
                        if ((int)lane == __ffs(peers) - 1) mat[sI * row + (p >> 5)] = (uint16_t)__popc(peers);
                    }
                }
            }
            bar_workers(G_THREADS);
            for (uint32_t sI = tid; sI < S; sI += G_THREADS) {  // suffix sums over the chunks of list sI
                uint16_t *mrow = mat + sI * row;
                uint32_t run = 0;
                for (int ch = (int)nch - 1; ch >= 0; ch--) {
                    const uint32_t c = mrow[ch];
                    mrow[ch] = (uint16_t)run;
                    run += c;
                }
            }
            bar_workers(G_THREADS);
#pragma unroll
            for (int it = 0; it < ITERS; it++) {
                const uint32_t p = it * G_THREADS + tid;
                const uint32_t sI = p < n_inst ? grp[p] : 0xFFFFu;
                if (sI != 0xFFFFu) {
                    const uint32_t a = arr[p];
                    out.stg_ids[idb + off[sI] + mat[sI * row + (p >> 5)] + within[it]] = ids_by_arrival ? ids_by_arrival[a] : id_base + (int32_t)a;
                }
            }
        } else {
            // ---- id lists, general path (slices of a big bucket, or very many lists): stage the arrivals of every list
            // in the order the grouping happened to rank them, then every instance finds its place by counting the
            // larger arrivals of its list (ties — the same read twice — by staging position).
            for (uint32_t i = tid; i < n_inst; i += G_THREADS) {
                const uint32_t sI = grp[i];
                if (sI != 0xFFFFu) stage_ids[off[sI] + rnk[i]] = arr[i];
            }
            bar_workers(G_THREADS);
            for (uint32_t i = tid; i < n_inst; i += G_THREADS) {
                const uint32_t sI = grp[i];
                if (sI == 0xFFFFu) continue;
                const uint32_t o = off[sI], c = (sI + 1 < S ? off[sI + 1] : N) - o, a = arr[i], r = rnk[i];
                const uint32_t *lst = stage_ids + o;
                uint32_t rank = 0;
                for (uint32_t y = 0; y < r; y++) rank += lst[y] >= a ? 1u : 0u;  // earlier staging position wins a tie
                for (uint32_t y = r + 1; y < c; y++) rank += lst[y] > a ? 1u : 0u;
                out.stg_ids[idb + o + rank] = ids_by_arrival ? ids_by_arrival[a] : id_base + (int32_t)a;
            }
        }

        // ---- stage the unit's slice of the flat table
        for (uint32_t x = tid; x < S; x += G_THREADS) {
            const uint32_t i = surv[x];
            const uint64_t q = (uint64_t)kb + x;
            out.stg_codes[q * KW] = key0[i];
            if (KW == 2) out.stg_codes[q * KW + 1] = key1[i];
            out.stg_mmer[q] = mm[i];
            out.stg_off[q] = off[x];
        }
        __threadfence();  // the staged unit is read back through L2 by the control warp (ld.cg): make the stores visible there first
        bar_all();        // Y: the unit is staged
        have_prev = true;
        prev_u = u;
        prev_S = S;
        prev_N = N;
        prev_idb = idb;
        prev_kb = kb;
    }
    // ---- the last unit of this CTA
    if (have_prev && ctrl) move_prev(resolve_prev());
}

// ------------------------------------------------------------------ bucket directory from the emitted k-mers

struct KmerBucketHead {
    const uint32_t *kmer_mmer;
    __device__ __forceinline__ uint32_t operator()(uint64_t s) const { return (s == 0 || kmer_mmer[s] != kmer_mmer[s - 1]) ? 1u : 0u; }
};

__global__ void emit_buckets_kernel(const uint32_t *__restrict__ kmer_mmer, const uint32_t *__restrict__ bucket_excl, uint64_t n_kmers,
                                    uint64_t n_ids, uint32_t *__restrict__ mmer_codes, uint64_t *__restrict__ mmer_kmer_off,
                                    uint64_t *__restrict__ kmer_id_off) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_kmers) return;
    const uint32_t head = KmerBucketHead{kmer_mmer}(s);
    if (head) {
        mmer_codes[bucket_excl[s]] = kmer_mmer[s];
        mmer_kmer_off[bucket_excl[s]] = s;
    }
    if (s == n_kmers - 1) {
        mmer_kmer_off[bucket_excl[s] + head] = n_kmers;
        kmer_id_off[n_kmers] = n_ids;
    }
}

__global__ void empty_table_kernel2(uint64_t *mmer_kmer_off, uint64_t *kmer_id_off) {
    mmer_kmer_off[0] = 0;
    kmer_id_off[0] = 0;
}

// ------------------------------------------------------------------ host side

static PlanParams plan_params() { return PlanParams{G_UNIT_CAP, G_UNIT_CAP / 2, G_UNIT_CAP / 2, G_UNIT_CAP / 2}; }

static size_t skr_group_smem_bytes(int KW) {
    const size_t cap = G_UNIT_CAP;
    const size_t hs = cap > 2048 ? 8192 : (cap > 1024 ? 4096 : 2048);  // hash slots, as in the kernel
    return KW * cap * 8 + cap * 4 * 2 + hs * 4 + cap * 4 + cap * 2 * 3 + 64;
}


// Phase A (needs n_skr on the host): instance prefix and m-mer run starts in one fused scan.
// both64: [n_skr + 1] u64 scratch; scratch64: prefix-scan scratch. *n_inst_dev / *n_runs_dev receive the totals.
static int skr_plan_runs(const uint64_t *side, uint64_t n_skr, uint32_t *inst_prefix /*[n+1]*/, uint64_t *both64, uint32_t *run_start /*[n+1]*/,
                  uint64_t *scratch64, uint32_t *n_inst_dev, uint32_t *n_runs_dev, cudaStream_t st) {
    int l = exclusive_scan<uint64_t, SkrCountAndHead>(SkrCountAndHead{side}, both64, n_skr, scratch64, both64 + n_skr, st);
    skr_run_starts_kernel<<<(unsigned)((n_skr + 255) / 256), 256, 0, st>>>(side, n_skr, both64, both64 + n_skr, inst_prefix, run_start, n_inst_dev,
                                                                          n_runs_dev);
    return l + 1;
}

// Phase B (needs n_runs on the host): units. small_prefix / unit_base are [n_runs] scratch arrays.
static int skr_plan_units(const void *skr_sorted, int K, const uint32_t *inst_prefix, const uint32_t *run_start, uint64_t n_runs,
                   uint32_t *small_prefix, uint32_t *unit_base, uint32_t *scratch, void *units, uint64_t max_units, void *gc_dev,
                   uint32_t *big_list, uint64_t *big_k0, uint64_t *big_k1, uint32_t *big_arr, int sm_count, cudaStream_t st) {
    RunView rv{run_start, inst_prefix};
    const PlanParams pp = plan_params();
    GroupCounters *gc = static_cast<GroupCounters *>(gc_dev);
    int l = 0;
    cudaMemsetAsync(units, 0, sizeof(Unit) * max_units, st);
    cudaMemsetAsync(gc, 0, sizeof(GroupCounters), st);
    l += exclusive_scan<uint32_t, SmallSize>(SmallSize{rv, pp}, small_prefix, n_runs, scratch, nullptr, st);
    l += exclusive_scan<uint32_t, UnitsOfRun>(UnitsOfRun{rv, small_prefix, pp}, unit_base, n_runs, scratch, &gc->n_units, st);
    fill_units_kernel<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(rv, small_prefix, unit_base, n_runs, pp, static_cast<Unit *>(units), gc,
                                                                       big_list);
    const unsigned grid = (unsigned)sm_count * 6;
    const size_t part_smem = (size_t)PART_SAMPLES * 8 + (size_t)PART_FINE * 8 + (size_t)PART_FINE * 4 + ((size_t)PART_FINE + 1) * 4;
    const uint32_t *s = static_cast<const uint32_t *>(skr_sorted);
    BigScratch sc{big_k0, big_k1, big_arr};
    if (K <= 32) {
        cudaFuncSetAttribute(partition_big_runs_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)part_smem);
        partition_big_runs_kernel<2, 1><<<grid, PART_THREADS, part_smem, st>>>(s, rv, unit_base, big_list, gc, pp, K, sc, static_cast<Unit *>(units));
    } else {
        cudaFuncSetAttribute(partition_big_runs_kernel<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)part_smem);
        partition_big_runs_kernel<4, 2><<<grid, PART_THREADS, part_smem, st>>>(s, rv, unit_base, big_list, gc, pp, K, sc, static_cast<Unit *>(units));
    }
    return l + 2;
}

// After chunk `chunk` of the grouping has completed: its end offsets {surviving k-mers << 31 | ids} = the inclusive prefix of
// its last unit (every unit of the chunk has resolved by then).  An empty prefix of the unit list yields 0.
__global__ void publish_chunk_total_kernel(const unsigned long long *__restrict__ unit_state, const GroupCounters *__restrict__ gc, uint32_t chunk,
                                           uint32_t n_chunks, unsigned long long *__restrict__ chunk_totals) {
    const uint32_t end = (uint32_t)(((uint64_t)gc->n_units * (chunk + 1)) / n_chunks);
    chunk_totals[chunk] = end ? (unit_state[end - 1] & LKB_VALUE_MASK) : 0ull;
}

int run_v2_group(gbin_ctx *ctx, void *skr, void *twin, uint64_t n_skr, const int32_t *d_ids, int32_t id_base, cudaStream_t st, gbin_table *out,
                 int *launches, bool *done, uint64_t *n_inst_out, HostSink *sink) {
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
    const uint64_t max_units = n / (G_UNIT_CAP / 4) + 2 * n_runs + 8;
    CU(ctx->small_prefix.ensure((n_runs + 1) * 4));
    CU(ctx->unit_base.ensure((n_runs + 1) * 4));
    CU(ctx->units.ensure(max_units * sizeof(Unit)));
    CU(ctx->unit_state.ensure(max_units * 8));
    CU(ctx->big_list.ensure((n / (uint64_t)G_UNIT_CAP + 2) * 8));  // buckets larger than a unit
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
    // The grouping runs as n_ch consecutive launches over equal ranges of the unit list, one chained scan across them.  On the host
    // path the end offsets of every chunk ({k-mers << 31 | ids}) are published after it, so that finished parts of the table stream out.
    const bool stream = sink && sink->chunks > 1;
    const uint32_t n_ch = stream ? (uint32_t)sink->chunks : 1u;
    const size_t smem = skr_group_smem_bytes(KW);
    on = ctx->prof.begin(KK_SKR_GROUP, st);
    unsigned long long *unit_state = ctx->unit_state.as<unsigned long long>();
    cudaMemsetAsync(unit_state, 0, sizeof(unsigned long long) * max_units, st);
    cudaMemsetAsync(dm->chunk_tickets, 0, sizeof(uint32_t) * n_ch, st);
    const GroupOut go{ctx->o_kmer_codes.as<uint64_t>(), ctx->o_kmer_mmer.as<uint32_t>(), ctx->o_kmer_id_off.as<uint64_t>(), ctx->o_read_ids.as<int32_t>(), kmer_cap,
                      n, ctx->stg_ids.as<int32_t>(), ctx->stg_codes.as<uint64_t>(), ctx->stg_mmer.as<uint32_t>(), ctx->stg_off.as<uint32_t>()};
    const BigScratch big{ctx->big_k0.as<uint64_t>(), ctx->big_k1.as<uint64_t>(), ctx->big_arr.as<uint32_t>()};
    auto launch = [&](auto kern, int threads, int ctas_per_sm) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        for (uint32_t c = 0; c < n_ch; c++) {
            kern<<<ctx->sm_count * ctas_per_sm, threads + 32, smem, st>>>(static_cast<const uint32_t *>(sorted), ctx->inst_prefix.as<uint32_t>(),
                                                                          ctx->units.as<Unit>(), big, K, cutoff, d_ids, id_base, go, unit_state, &dm->gc, c,
                                                                          n_ch, dm->chunk_tickets);
            if (stream) {
                publish_chunk_total_kernel<<<1, 1, 0, st>>>(unit_state, &dm->gc, c, n_ch, dm->chunk_totals);
                cudaMemcpyAsync(hm->chunk_totals + c, dm->chunk_totals + c, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
                cudaEventRecord(ctx->ev_chunk[c], st);
            }
        }
    };
    const int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));  // CTAs per SM that shared memory allows
    if (KW == 1) launch(skr_group_kernel<2, 1, G_UNIT_CAP, 256>, 256, per_sm < 4 ? per_sm : 4);
    else launch(skr_group_kernel<4, 2, G_UNIT_CAP, 256>, 256, per_sm < 4 ? per_sm : 4);
    lp = (int)(stream ? 2 * n_ch : n_ch);
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    if (stream) {
        const int rc = stream_finished_chunks(ctx, sink, n_ch, hm->chunk_totals, 31, nullptr);
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

int emit_bucket_directory(gbin_ctx *ctx, uint64_t S, uint64_t NS, cudaStream_t st, int *launches, uint64_t *B) {
    Misc *dm = ctx->misc.as<Misc>();
    Misc *hm = static_cast<Misc *>(ctx->h_misc.p);
    CU(ctx->bucket_excl.ensure((S + 1) * 4));
    CU(ctx->o_mmer_codes.ensure((S + 1) * sizeof(uint32_t)));
    CU(ctx->o_mmer_kmer_off.ensure((S + 2) * sizeof(uint64_t)));
    CU(ctx->scan_scratch.ensure(group_scan_scratch_bytes(S + 1024)));
    const bool on = ctx->prof.begin(KK_EMIT, st);
    int lp = 1;
    if (S == 0) {
        cudaMemsetAsync(&dm->n_buckets_dev, 0, sizeof(uint32_t), st);
        empty_table_kernel2<<<1, 1, 0, st>>>(ctx->o_mmer_kmer_off.as<uint64_t>(), ctx->o_kmer_id_off.as<uint64_t>());
    } else {
        const uint32_t *kmer_mmer = ctx->o_kmer_mmer.as<uint32_t>();
        lp += exclusive_scan<uint32_t, KmerBucketHead>(KmerBucketHead{kmer_mmer}, ctx->bucket_excl.as<uint32_t>(), S, ctx->scan_scratch.as<uint32_t>(),
                                                       &dm->n_buckets_dev, st);
        emit_buckets_kernel<<<(unsigned)((S + 255) / 256), 256, 0, st>>>(kmer_mmer, ctx->bucket_excl.as<uint32_t>(), S, NS, ctx->o_mmer_codes.as<uint32_t>(),
                                                                        ctx->o_mmer_kmer_off.as<uint64_t>(), ctx->o_kmer_id_off.as<uint64_t>());
    }
    ctx->prof.end(on, lp, st);
    *launches += lp;
    CU(cudaGetLastError());
    CU(read_back(ctx, &Misc::n_buckets_dev, st));
    *B = hm->n_buckets_dev;
    return GBIN_OK;
}

}  // namespace gbin
