// bin3.cuh — pipeline v3: shared definitions (key layout, pieces, units, chained-scan state).
//
// v3 keeps the super-k-mer records of the scan stage where they are and sorts 8-byte *entries* {key << 32 | slot} that
// refer to them ("sort by reference").  An entry stands for a *piece* of a record: the windows of one d-class, where
// d = so - t is the offset of the signature m-mer inside window t's k-mer (0 <= d <= K-M).  d is a function of
// (m-mer code, oriented k-mer): the signature is the leftmost position of the k-mer whose score reaches the bucket's
// code (binning.c:922 keeps a signature until the window start passes it, :972 replaces it only on a strictly larger
// score, so no position of the k-mer before the signature scores as high).  Equal keys therefore have equal d, and
// instances with different d can be grouped independently.
//   nc == 1: one piece per record (all windows), key = m-mer code.
//   nc == 2: class 0 = windows with d >= d0, class 1 = windows with d < d0; with h > 0 the key is extended by the h
//            oriented bases next to the signature that every k-mer of the class contains (left of it for class 0,
//            right of it for class 1): key = mmer << (1 + 2h) | class << 2h | flank.  Level 2 of the store then
//            breaks into sub-buckets of one locus each even when an m-mer bucket holds thousands of loci.
#pragma once
#include <cstdint>

#include "skr.cuh"

namespace gbin {

struct KeyLayout {
    int K, M;
    int h;         // flank bases in the key (0 = none)
    int nc;        // pieces per record: 1 or 2
    int d0;        // class 1 iff d < d0 (nc == 2)
    int cshift;    // log2(nc): slot = record << cshift | class
    int mshift;    // key >> mshift = m-mer code
    int key_bits;  // bits of the key that take part in the sort (one more than the widest real key when nc == 2, so that
                   // the all-ones key of an empty piece sorts behind everything)
};

__host__ __device__ inline KeyLayout make_key_layout(int K, int M, int h, int nc) {
    KeyLayout kl;
    kl.K = K;
    kl.M = M;
    if (nc != 2) {
        nc = 1;
        h = 0;
    }
    const int span = K - M + 1;  // d values
    kl.d0 = (span + 1) / 2;
    if (nc == 2) {
        // class 0 needs d >= h for all its windows (d >= d0), class 1 needs K-M-d >= h for all its windows (d <= d0-1)
        int hmax = kl.d0 < (K - M - (kl.d0 - 1)) ? kl.d0 : (K - M - (kl.d0 - 1));
        while (2 * M + 1 + 2 * hmax > 31) hmax--;
        if (hmax < 0) hmax = 0;
        if (h > hmax) h = hmax;
        if (h < 0) h = 0;
        if (2 * M + 1 > 31) {  // no room for the class bit: fall back to one piece per record
            nc = 1;
            h = 0;
        }
    }
    kl.h = h;
    kl.nc = nc;
    kl.cshift = nc == 2 ? 1 : 0;
    kl.mshift = nc == 2 ? 1 + 2 * h : 0;
    kl.key_bits = nc == 2 ? 2 * M + 1 + 2 * h + 1 : 2 * M;
    return kl;
}

// Windows [t0, t0 + np) of a record (header word 2 = n | rev << 8 | so << 16) that belong to class `cls`.
__host__ __device__ inline void piece_of(uint32_t meta, uint32_t cls, const KeyLayout &kl, uint32_t *t0, uint32_t *np) {
    const uint32_t n = meta & 0xffu;
    const int so = (int)((meta >> 16) & 0xffu);
    if (kl.nc == 1) {
        *t0 = 0;
        *np = n;
    } else if (cls == 0) {  // d >= d0  <=>  t <= so - d0
        const int last = so - kl.d0;
        *t0 = 0;
        *np = last < 0 ? 0u : ((uint32_t)last + 1u < n ? (uint32_t)last + 1u : n);
    } else {  // d < d0  <=>  t >= so - d0 + 1
        const int first = so - kl.d0 + 1 > 0 ? so - kl.d0 + 1 : 0;
        *t0 = (uint32_t)first;
        *np = n > (uint32_t)first ? n - (uint32_t)first : 0u;
    }
}

// One unit of the grouping kernel = one warp's worth of work.
//   packed unit: whole atoms (runs of equal key) [ent_begin, ent_end) of the sorted entries, n_inst <= capacity;
//   round unit : round `round` of `rounds` over ONE atom that is larger than the capacity: the atom's instances are cut
//                by ranges of d (chosen by the planner from the atom's d-histogram), every round groups one range.
// A bucket (all atoms of one m-mer code) that does not fit one unit is a *span* of consecutive units that hold nothing else;
// its k-mers come out unit by unit, each unit ascending: the finalize pass merges them into one ascending run.
struct __align__(16) Unit3 {
    uint32_t ent_begin, ent_end;
    uint32_t n_inst;         // instances of the unit (round units: of the atom until the planner has cut it, then of the round)
    uint32_t round, rounds;  // rounds == 0: packed unit
    uint32_t drange;         // round units: dlo | dhi << 8
    uint32_t ibase;          // instance coordinate of the unit's first instance
    uint32_t span_len;       // 0: the unit holds whole buckets; L: first of the L units of a bucket that does not fit one unit; ~0: another unit of such a bucket
};

// Device scalars of pipeline 3 (the host reads them through Misc::gc3).
struct G3Counters {
    unsigned long long distinct;
    unsigned long long total_kmers, total_ids;
    unsigned int overflow;
    unsigned int n_units, n_spans;
    unsigned int pad;
    unsigned long long lsd_kmers, lsd_ids;  // surviving k-mers / ids of the spans that are put in order by the global sort
};

}  // namespace gbin
