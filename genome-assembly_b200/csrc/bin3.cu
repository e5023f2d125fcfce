// bin3.cu — pipeline v3: level 1 by reference, level 2 by one warp (or one pair of warps) per unit.
//
// Input: the super-k-mer records of the scan stage, in arrival order (skr.cuh).  Stages:
//   1. make_entries_kernel: one 8-byte entry {key << 32 | slot} per piece of a record (bin3.cuh) and the piece's
//      window count (one byte per slot).  The records themselves never move again.
//   2. radix_sort_entries (radix_sort.cu): stable LSD sort of the entries on the key = level 1 of the reference's
//      two-level store (binning.c:1044-1049); inside a key entries stay in arrival order.
//   3. planning (no atomics, no host round trip inside): instance prefix + atoms (runs of equal key) in one scan;
//      units = packs of whole small atoms, single atoms, or the d-rounds of an atom larger than a unit.
//   4. group3_kernel: every WARP (512-instance units) or PAIR of warps (1024-instance units, synchronised by the pair's own
//      named barrier) owns one unit at a time — no CTA barrier anywhere.  It expands the windows of its pieces (rolling
//      2-bit shift, complement when is_rev — binning.c:1029-1040) into shared memory, groups equal (bucket, k-mer) keys with a hash whose slots hold instance indices (level-2 insert + ll_node push,
//      binning.c:1052-1069), counts, prunes (count > ABUNDANCE_CUTOFF, binning.c:1094-1102), orders the survivors of
//      every bucket by k-mer, orders every id list newest-first, obtains its place in the table from a two-level chained
//      scan over units (aggregates are published right after the count, long before they are needed) and writes its part
//      of the flat table ONCE, at its final place.
//   5. span_reorder_kernel: atoms that were split into d-rounds come out round by round; their (few) surviving k-mers
//      are sorted and their id lists moved from the staging arrays to the final place.
//   6. skr_emit_buckets (skr_group.cu): bucket directory; buckets that lost all k-mers vanish (binning.c:1136-1142).
#include "bin3.cuh"
#include "gbin_device.cuh"
#include "gbin_internal.h"
#include "prefix_scan.cuh"

namespace gbin {

// ------------------------------------------------------------------ entries

// h oriented bases starting at base j of the payload (2 bits per base, MSB first, 16 bases per u32 word).
__device__ __forceinline__ uint32_t payload_bases(const uint32_t *pl, uint32_t nwords, uint32_t j, uint32_t h, bool rev) {
    const uint32_t bit = 2 * j, wi = bit >> 5, sh = bit & 31;
    const uint32_t a = wi < nwords ? pl[wi] : 0u, b = wi + 1 < nwords ? pl[wi + 1] : 0u;
    uint32_t x = __funnelshift_l(b, a, sh);  // 16 bases starting at j
    if (rev) x = ~x;
    return h ? (x >> (32 - 2 * h)) : 0u;
}

template <int PW>
__global__ void __launch_bounds__(256)
    make_entries_kernel(const uint32_t *__restrict__ skr, uint64_t n_rec, KeyLayout kl, uint64_t *__restrict__ ent, uint16_t *__restrict__ piece_info,
                        unsigned long long *__restrict__ n_real) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t real = 0;
    if (i < n_rec) {
        const uint4 h = *reinterpret_cast<const uint4 *>(skr + i * NW);
        const uint32_t mmer = h.y, meta = h.z;
        if (kl.nc == 1) {
            ent[i] = ((uint64_t)mmer << 32) | (uint32_t)i;
            const uint32_t n = meta & 0xffu, so1 = (meta >> 16) & 0xffu;
            piece_info[i] = (uint16_t)(n | ((so1 - (n - 1)) << 8));  // windows | smallest d of the piece << 8
            real = 1;
        } else {
            const bool rev = (meta >> 8) & 1u;
            const uint32_t so = (meta >> 16) & 0xffu;
            const uint32_t *pl = skr + i * NW + 4;
#pragma unroll
            for (uint32_t c = 0; c < 2; c++) {
                uint32_t t0, np;
                piece_of(meta, c, kl, &t0, &np);
                const uint32_t slot = (uint32_t)(2 * i + c);
                uint32_t key = 0xffffffffu;
                if (np) {
                    const uint32_t fl = kl.h ? payload_bases(pl, 2 * PW, c == 0 ? so - kl.h : so + kl.M, kl.h, rev) : 0u;
                    key = (mmer << kl.mshift) | (c << (2 * kl.h)) | fl;
                    real++;
                }
                ent[slot] = ((uint64_t)key << 32) | slot;
                piece_info[slot] = (uint16_t)(np | (np ? (so - (t0 + np - 1)) << 8 : 0u));
            }
        }
    }
    if (kl.nc == 1) return;  // every slot is real: the host knows the count
    __shared__ uint32_t s_real;
    if (threadIdx.x == 0) s_real = 0;
    __syncthreads();
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) real += __shfl_xor_sync(0xffffffffu, real, d);
    if ((threadIdx.x & 31) == 0 && real) atomicAdd(&s_real, real);
    __syncthreads();
    if (threadIdx.x == 0 && s_real) atomicAdd(n_real, (unsigned long long)s_real);
}

int v3_make_entries(const void *skr, uint64_t n_rec, const KeyLayout &kl, uint64_t *ent, uint16_t *piece_info, unsigned long long *n_real_dev,
                    cudaStream_t st) {
    cudaMemsetAsync(n_real_dev, 0, sizeof(unsigned long long), st);
    if (n_rec == 0) return 0;
    const unsigned grid = (unsigned)((n_rec + 255) / 256);
    if (kl.K <= 32) make_entries_kernel<2><<<grid, 256, 0, st>>>(static_cast<const uint32_t *>(skr), n_rec, kl, ent, piece_info, n_real_dev);
    else make_entries_kernel<4><<<grid, 256, 0, st>>>(static_cast<const uint32_t *>(skr), n_rec, kl, ent, piece_info, n_real_dev);
    return 1;
}

// ------------------------------------------------------------------ planning

struct EntCountAndHead {  // low half: windows of sorted entry i; high half: 1 if it starts a new atom (run of equal key)
    const uint64_t *ent;
    const uint16_t *info;  // per sorted entry: windows | smallest d << 8 (gathered by the last sort pass)
    __device__ __forceinline__ uint64_t operator()(uint64_t i) const {
        const uint64_t e = ent[i];
        const uint64_t head = (i == 0 || (e >> 32) != (ent[i - 1] >> 32)) ? 1ull : 0ull;
        return (uint64_t)(info[i] & 0xffu) | (head << 32);
    }
};

struct EntRunSink {  // consumer of the scan above: instance prefix of every sorted entry, first entry of every atom
    const uint64_t *ent;
    uint32_t *inst_prefix, *run_start;
    __device__ __forceinline__ void operator()(uint64_t i, uint64_t b) const {
        inst_prefix[i] = (uint32_t)b;
        if (i == 0 || (ent[i] >> 32) != (ent[i - 1] >> 32)) run_start[b >> 32] = (uint32_t)i;
    }
};

__global__ void v3_run_totals_kernel(const uint64_t *__restrict__ total, uint64_t n, uint32_t *__restrict__ inst_prefix, uint32_t *__restrict__ run_start,
                                     uint32_t *__restrict__ n_inst_out, uint32_t *__restrict__ n_runs_out) {
    const uint64_t t = *total;
    inst_prefix[n] = (uint32_t)t;
    run_start[t >> 32] = (uint32_t)n;
    *n_inst_out = (uint32_t)t;
    *n_runs_out = (uint32_t)(t >> 32);
}

int v3_plan_runs(const uint64_t *ent, const uint16_t *sorted_info, uint64_t n_ent, uint32_t *inst_prefix, uint64_t *both64, uint32_t *run_start,
                 uint64_t *scratch64, uint32_t *n_inst_dev, uint32_t *n_runs_dev, cudaStream_t st) {
    if (n_ent == 0) {
        cudaMemsetAsync(n_inst_dev, 0, 4, st);
        cudaMemsetAsync(n_runs_dev, 0, 4, st);
        return 0;
    }
    int l = exclusive_scan_to<uint64_t, EntCountAndHead, EntRunSink>(EntCountAndHead{ent, sorted_info}, EntRunSink{ent, inst_prefix, run_start}, n_ent, scratch64,
                                                                     both64, st);
    v3_run_totals_kernel<<<1, 1, 0, st>>>(both64, n_ent, inst_prefix, run_start, n_inst_dev, n_runs_dev);
    return l + 1;
}

// Packing: a unit is a run of consecutive atoms (so that unit order is key order) with at most `cap` instances, NB atoms
// and EC entries — chosen greedily: an atom joins the current unit if it still fits, else it opens the next one.  Greedy
// packing is a sequential recurrence; it is made parallel by restarting it at every block of PLAN_BLOCK atoms (one extra
// partial unit per block, under 2 % of the units).  An atom with more than `cap` instances gets 2 * ceil(c / cap) + 1
// round units (enough for a greedy cut of its d-histogram whenever no single d holds more than cap instances).
constexpr int PLAN_BLOCK = 64;    // atoms walked by one thread
struct Plan3 {
    uint32_t cap, nb_max, ecap, max_rounds;
    // limits for packing several buckets into one unit (<= the limits above).  With cap = 1024 and two grouping kernels these are
    // the limits of the 512-instance kernel: small buckets share small units, a bucket between the two sizes is a unit of its own.
    uint32_t cap_s, nb_s, ecap_s;
};
struct RunView3 {
    const uint32_t *run_start;    // [NR+1]
    const uint32_t *inst_prefix;  // [E+1]
    __device__ __forceinline__ uint32_t size(uint64_t r) const { return inst_prefix[run_start[r + 1]] - inst_prefix[run_start[r]]; }
};
__host__ __device__ inline uint32_t rounds_of(uint32_t c, const Plan3 &pp) {
    uint32_t r = 2 * ((c + pp.cap - 1) / pp.cap) + 1;
    return r < pp.max_rounds ? r : pp.max_rounds;
}

// Per atom (run of equal key): instances, entries and m-mer code, for the packer.
__global__ void v3_atoms_kernel(RunView3 rv, const uint64_t *__restrict__ ent, uint64_t n_runs, int mshift, uint32_t *__restrict__ atom_c,
                                uint32_t *__restrict__ atom_e, uint32_t *__restrict__ atom_mm) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint32_t a = rv.run_start[r], b = rv.run_start[r + 1];
    atom_c[r] = rv.inst_prefix[b] - rv.inst_prefix[a];
    atom_e[r] = b - a;
    atom_mm[r] = (uint32_t)(ent[a] >> 32) >> mshift;
}

// nunits[r] = units that start at atom r (low half) | ATOM_ROUNDS if the atom is split into rounds.
// spanlen[r] = 0: the atom's bucket fits a unit; L > 0 at the first atom of a bucket that is a span of L units; SPAN_MEMBER at the
// other atoms of such a bucket.  A bucket (run of atoms with one m-mer code) is packed whole when it fits a unit; otherwise it
// becomes a span: units that hold nothing but this bucket — its atoms packed greedily, atoms larger than a unit cut into rounds.
// One thread walks PLAN_BLOCK atoms' worth of buckets: from the first bucket that starts at or after its block to the end of the
// bucket that straddles the block's end.
constexpr uint64_t ATOM_ROUNDS = 1ull << 32;
constexpr uint32_t SPAN_MEMBER = 0xfffffffeu;       // a further unit of a short span (merged by the warp of its first unit)
constexpr uint32_t SPAN_MEMBER_LONG = 0xffffffffu;  // a unit of a long span (put in order by the global sort)
constexpr uint32_t SPAN_SHORT_MAX = 17;             // units of a short span (an atom of up to 8 units' worth of instances gets 2 * 8 + 1 round units)
__global__ void __launch_bounds__(128)
    v3_pack_kernel(const uint32_t *__restrict__ atom_c, const uint32_t *__restrict__ atom_e, const uint32_t *__restrict__ atom_mm, uint64_t n_runs, Plan3 pp,
                   uint64_t *__restrict__ nunits, uint32_t *__restrict__ spanlen) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t r = t * PLAN_BLOCK;
    const uint64_t stop = r + PLAN_BLOCK < n_runs ? r + PLAN_BLOCK : n_runs;
    if (r >= n_runs) return;
    if (r > 0)
        while (r < n_runs && atom_mm[r] == atom_mm[r - 1]) r++;  // that bucket belongs to the previous walker
    uint32_t cur_c = 0, cur_e = 0, cur_b = 0;
    while (r < stop) {
        const uint32_t mm = atom_mm[r];
        uint64_t q = r;
        uint64_t cb = 0, eb = 0;
        do {
            cb += atom_c[q];
            eb += atom_e[q];
            q++;
        } while (q < n_runs && atom_mm[q] == mm);
        if (cb <= pp.cap && eb <= pp.ecap) {  // the whole bucket is one item
            if (cb > pp.cap_s || eb > pp.ecap_s) {  // too large to share a unit
                nunits[r] = 1ull;
                cur_b = 0;  // the next bucket opens a unit
            } else if (cur_b == 0 || cur_c + cb > pp.cap_s || cur_e + eb > pp.ecap_s || cur_b + 1 > pp.nb_s) {
                nunits[r] = 1ull;
                cur_c = (uint32_t)cb;
                cur_e = (uint32_t)eb;
                cur_b = 1;
            } else {
                nunits[r] = 0ull;
                cur_c += (uint32_t)cb;
                cur_e += (uint32_t)eb;
                cur_b++;
            }
            spanlen[r] = 0;
            for (uint64_t a = r + 1; a < q; a++) {
                nunits[a] = 0ull;
                spanlen[a] = 0;
            }
        } else {  // a span
            cur_b = 0;  // the next bucket opens a unit
            uint32_t L = 0, sc = 0, se = 0;
            bool open = false;
            for (uint64_t a = r; a < q; a++) {
                const uint32_t c = atom_c[a], e = atom_e[a];
                if (c > pp.cap) {
                    const uint32_t R = rounds_of(c, pp);
                    nunits[a] = (uint64_t)R | ATOM_ROUNDS;
                    L += R;
                    open = false;
                } else if (!open || sc + c > pp.cap || se + e > pp.ecap) {
                    nunits[a] = 1ull;
                    L++;
                    sc = c;
                    se = e;
                    open = true;
                } else {
                    nunits[a] = 0ull;
                    sc += c;
                    se += e;
                }
                spanlen[a] = SPAN_MEMBER;
            }
            spanlen[r] = L;
            if (L > SPAN_SHORT_MAX)
                for (uint64_t a = r + 1; a < q; a++) spanlen[a] = SPAN_MEMBER_LONG;
        }
        r = q;
    }
}

struct G3Counters {
    unsigned long long distinct;
    unsigned long long total_kmers, total_ids;
    unsigned int overflow;
    unsigned int n_units, n_spans;
    unsigned int pad;
    unsigned long long lsd_kmers, lsd_ids;  // surviving k-mers / ids of the spans that are put in order by the global sort
};

__global__ void v3_head_runs_kernel(const uint64_t *__restrict__ nunits, const uint64_t *__restrict__ base, uint64_t n_runs, uint32_t *__restrict__ head_run) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint32_t nu = (uint32_t)nunits[r];
    const uint32_t ub = (uint32_t)base[r];
    for (uint32_t j = 0; j < nu; j++) head_run[ub + j] = (uint32_t)r;
}

__global__ void v3_fill_units_kernel(RunView3 rv, const uint64_t *__restrict__ nunits, const uint32_t *__restrict__ spanlen, const uint64_t *__restrict__ base,
                                     const uint64_t *__restrict__ totals, uint64_t n_runs, const uint32_t *__restrict__ head_run, Unit3 *__restrict__ units,
                                     G3Counters *__restrict__ gc) {
    const uint32_t n_units = (uint32_t)*totals;
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u == 0) {
        gc->n_units = n_units;
        gc->n_spans = (uint32_t)(*totals >> 32);
    }
    if (u >= n_units) return;
    const uint32_t r0 = head_run[u];
    const uint64_t nu = nunits[r0];
    const uint32_t ub = (uint32_t)base[r0];
    Unit3 un;
    un.drange = 0u | (63u << 8);
    un.ent_begin = rv.run_start[r0];
    un.ibase = rv.inst_prefix[un.ent_begin];
    if (nu & ATOM_ROUNDS) {
        un.ent_end = rv.run_start[r0 + 1];
        un.n_inst = rv.inst_prefix[un.ent_end] - un.ibase;
        un.round = u - ub;
        un.rounds = (uint32_t)nu;
    } else {
        const uint32_t r1 = (u + 1 < n_units) ? head_run[u + 1] : (uint32_t)n_runs;
        un.ent_end = rv.run_start[r1];
        un.n_inst = rv.inst_prefix[un.ent_end] - un.ibase;
        un.round = 0;
        un.rounds = 0;
    }
    const uint32_t sl = spanlen[r0];
    // the head atom of a span carries its length; its first unit is the span's head, its further (round) units are members
    if (sl == 0 || sl == SPAN_MEMBER || sl == SPAN_MEMBER_LONG) un.span_len = sl;
    else un.span_len = u == ub ? sl : (sl > SPAN_SHORT_MAX ? SPAN_MEMBER_LONG : SPAN_MEMBER);
    units[u] = un;
}

// One warp per split atom: d-histogram of the atom (difference array over its pieces, then prefix), greedy cut into rounds of
// consecutive d whose instances fit a unit.  Fills the atom's round units: d-range, instance coordinate, instances (0 = unused).
__global__ void __launch_bounds__(128)
    v3_round_cuts_kernel(const uint16_t *__restrict__ info, Unit3 *__restrict__ units, G3Counters *__restrict__ gc, uint32_t cap) {
    __shared__ int s_hist[4][68];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int *dhist = s_hist[warp];
    const uint32_t n_units = gc->n_units;
    for (uint32_t u = blockIdx.x * 4 + warp; u < n_units; u += gridDim.x * 4) {
        const Unit3 un = units[u];
        if (un.rounds == 0 || un.round != 0) continue;
        dhist[lane] = 0;
        dhist[lane + 32] = 0;
        if (lane < 4) dhist[64 + lane] = 0;
        __syncwarp();
        const uint32_t n_ent = un.ent_end - un.ent_begin;
        for (uint32_t e = lane; e < n_ent; e += 32) {
            const uint32_t pi = info[un.ent_begin + e];
            const uint32_t np = pi & 0xffu, dlo = pi >> 8;
            if (np) {
                atomicAdd(&dhist[dlo], 1);        // smallest d of the piece
                atomicAdd(&dhist[dlo + np], -1);  // one past its largest d
            }
        }
        __syncwarp();
        const int a = dhist[2 * lane], b = dhist[2 * lane + 1];
        int incl = a + b;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += o;
        }
        __syncwarp();
        dhist[2 * lane] = incl - b;  // instances with d = 2 * lane
        dhist[2 * lane + 1] = incl;  // instances with d = 2 * lane + 1
        __syncwarp();
        if (lane == 0) {
            uint32_t rnd = 0, acc = 0, before = 0;
            int lo = 0;
            bool bad = false;
            auto emit = [&](int hi) {
                if (rnd < un.rounds) {
                    Unit3 &w = units[u + rnd];
                    w.drange = (uint32_t)lo | ((uint32_t)hi << 8);
                    w.ibase = un.ibase + before;
                    w.n_inst = acc;
                } else {
                    bad = true;
                }
            };
            for (int d = 0; d < 64; d++) {
                const uint32_t c = (uint32_t)dhist[d];
                if (c > cap) bad = true;
                if (acc + c > cap) {
                    emit(d - 1);
                    rnd++;
                    lo = d;
                    before += acc;
                    acc = 0;
                }
                acc += c;
            }
            emit(63);
            for (uint32_t j = rnd + 1; j < un.rounds; j++) {  // unused rounds
                units[u + j].n_inst = 0;
                units[u + j].ibase = un.ibase + un.n_inst;
            }
            if (bad) atomicExch(&gc->overflow, 1u);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------ the grouping kernel

struct UnitOut3 {  // what a unit reports: its place in the staging arrays and its totals
    uint32_t ibase;  // instance coordinate of the unit's first instance = where its ids are staged; its k-mers are staged at ibase / kdiv
    uint32_t S, N;   // surviving k-mers, ids
    uint32_t pad;
};

// Units never wait for each other: a unit writes its part of the table into staging arrays at a place that depends on the
// unit alone (ids at its instance coordinate, k-mers at that coordinate divided by cutoff + 1 — disjoint because a surviving
// k-mer has more than `cutoff` instances), and reports its totals.  One scan over the totals and finalize3_kernel then put
// everything at its final place.
struct G3Stage {
    uint64_t *codes;  // [kmer_cap * KW]
    uint32_t *mmer;   // [kmer_cap]
    uint32_t *loff;   // [kmer_cap] start of the k-mer's id list inside its unit
    int32_t *ids;     // [id_cap]
    UnitOut3 *unit_out;
    uint64_t kmer_cap, id_cap;
    uint32_t kdiv;
};

template <int PW>
struct Payload {
    uint64_t w[PW];
    __device__ __forceinline__ void set(const uint4 &a, const uint4 &b) {
        w[0] = ((uint64_t)a.x << 32) | a.y;
        w[1] = ((uint64_t)a.z << 32) | a.w;
        if (PW == 4) {
            w[PW - 2] = ((uint64_t)b.x << 32) | b.y;
            w[PW - 1] = ((uint64_t)b.z << 32) | b.w;
        }
    }
    __device__ __forceinline__ void advance(uint32_t bases) {  // 0 < 2 * bases < 64
        const uint32_t sh = 2 * bases;
#pragma unroll
        for (int q = 0; q < PW - 1; q++) w[q] = (w[q] << sh) | (w[q + 1] >> (64 - sh));
        w[PW - 1] <<= sh;
    }
    __device__ __forceinline__ void skip(uint32_t bases) {  // any number of bases
        while (bases >= 31) {
            advance(31);
            bases -= 31;
        }
        if (bases) advance(bases);
    }
};

// Oriented k-mer code of the window at the front of the payload (top 2K bits), complemented when rev (binning.c:1029-1040).
template <int PW, int KW>
__device__ __forceinline__ void front_kmer(const Payload<PW> &pl, int K, bool rev, uint64_t kmask0, uint64_t *k0, uint64_t *k1) {
    if (KW == 1) {
        uint64_t a = (2 * K == 64) ? pl.w[0] : (pl.w[0] >> (64 - 2 * K));
        if (rev) a = ~a & kmask0;
        *k0 = a;
        *k1 = 0;
    } else {
        const int r = 128 - 2 * K;  // 0..62
        uint64_t a = r ? (pl.w[0] >> r) : pl.w[0];
        uint64_t b = r ? ((pl.w[1] >> r) | (pl.w[0] << (64 - r))) : pl.w[1];
        if (rev) {
            a = ~a & kmask0;
            b = ~b;
        }
        *k0 = a;
        *k1 = b;
    }
}

template <int WCAP, int KW>
struct UnitLayout {  // shared memory of one unit in flight; every region is a multiple of 16 bytes
    static constexpr int W = WCAP == 1024 ? 2 : 1;  // warps per unit: one at 512 instances, a pair at 1024
    static constexpr int NB_MAX = WCAP / 8;  // buckets of a packed unit
    static constexpr int ECAP = WCAP / 4;    // entries of a packed unit (an atom with more entries is a unit of its own)
    static constexpr int BSTART_BYTES = ((NB_MAX + 1) * 2 + 15) / 16 * 16;
    static constexpr int XCH_BYTES = W == 2 ? 64 : 0;  // the pair's exchange words: [2 slots][2 warps][4] u32
    static constexpr int BYTES = KW * WCAP * 8 /*keys*/ + WCAP * 4 /*table*/ + W * WCAP * 2 /*cnt (+ cnt_lo)*/ + WCAP * 2 /*grp*/ + WCAP * 2 /*rk*/ + WCAP /*eix*/ +
                                 BSTART_BYTES + NB_MAX * 4 /*bmm*/ + ECAP * 4 /*eid*/ + ECAP /*ebk*/ + XCH_BYTES;
};

__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v, uint32_t lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= (uint32_t)d) v += o;
    }
    return v;
}

// Synchronises the warps of one unit: __syncwarp for one warp, the pair's own named barrier (bar.sync id, 64) for two — never the
// whole CTA, so a warp waits for its partner only.
template <int W>
__device__ __forceinline__ void unit_sync(uint32_t bar_id) {
    if (W == 1) __syncwarp();
    else asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
}

// A pair's exchange of warp-uniform values: lane 0 of every warp writes up to three values into the current slot, the pair syncs,
// and both warps read both sets (slot[0..2]: warp 0's, slot[4..6]: warp 1's).  Two slots are used in turn: a warp writes a slot again
// two exchanges later, after the barrier of the exchange in between, which its partner reaches only after reading that slot.
struct PairXch {
    uint32_t *x;
    uint32_t slot;
    __device__ __forceinline__ const uint32_t *put(uint32_t h, uint32_t lane, uint32_t bar_id, uint32_t a, uint32_t b = 0u, uint32_t c = 0u) {
        uint32_t *s = x + slot * 8;
        if (lane == 0) {
            s[h * 4] = a;
            s[h * 4 + 1] = b;
            s[h * 4 + 2] = c;
        }
        slot ^= 1u;
        unit_sync<2>(bar_id);
        return s;
    }
};

// Inclusive scan of v over the unit's 32 * W lanes (warp 1's lanes after warp 0's); *total = the sum over all of them.
template <int W>
__device__ __forceinline__ uint32_t unit_incl_scan(uint32_t v, uint32_t lane, uint32_t h, uint32_t bar_id, PairXch &xc, uint32_t *total) {
    v = warp_incl_scan_u32(v, lane);
    const uint32_t wt = __shfl_sync(0xffffffffu, v, 31);
    if (W == 1) {
        *total = wt;
        return v;
    }
    const uint32_t *s = xc.put(h, lane, bar_id, wt);
    *total = s[0] + s[4];
    return v + (h ? s[0] : 0u);
}

constexpr int G3_WARPS = 5;  // units in flight per CTA of the 512-instance layout (one warp each)
constexpr int G3_PAIRS = 3;  // units in flight per CTA of the 1024-instance layout (one pair of warps each): 3 CTAs, 18 warps per SM at K <= 32
// CTAs per SM that a CTA's shared memory allows (227 KB per SM, 1 KB of it reserved per CTA)
constexpr int g3_ctas_per_sm(size_t smem) {
    const int n = (int)((size_t)(227 * 1024) / (smem + 1024));
    return n > 1 ? n : 1;
}
constexpr uint32_t G3_SMALL_INST = 512, G3_SMALL_ENT = 128, G3_SMALL_NB = 64;  // what the 512-instance layout holds

// The pair kernel states the CTAs per SM that its shared memory allows, so that ptxas budgets registers for them (and keeps
// every value in a register); the one-warp kernel leaves the choice to ptxas.
template <int PW, int KW, int WCAP, int UNITS, int U>
__global__ void __launch_bounds__(UNITS * UnitLayout<WCAP, KW>::W * 32, WCAP == 1024 ? g3_ctas_per_sm(UNITS * UnitLayout<WCAP, KW>::BYTES) : 0)
    group3_kernel(const uint32_t *__restrict__ skr, const uint64_t *__restrict__ ent, const Unit3 *__restrict__ units, KeyLayout kl, int cutoff,
                  const int32_t *__restrict__ ids_by_arrival, int32_t id_base, G3Stage out, G3Counters *__restrict__ gc,
                  const uint32_t *__restrict__ chunk_bounds, uint32_t chunk, uint32_t *__restrict__ chunk_tickets, uint32_t size_class) {
    // size_class: 0 = every unit; 1 = only the small units (no rounds, at most G3_SMALL_INST instances and G3_SMALL_ENT entries);
    // 2 = only the others.  Two launches (1024-instance layout for the large units, 512-instance layout for the small ones) share
    // the unit list.
    // UNITS units are in flight per CTA.  A unit of the 512-instance layout is worked on by one warp; a unit of the 1024-instance
    // layout by a PAIR of warps that share its shared memory (h = 0, 1), synchronised by the pair's own named barrier: the unit's
    // memory fixes how many units an SM holds, not how many warps work on them.  The pair splits every phase: entries and
    // survivors by ranges of 64, the instance positions in two halves [0, mid) and [mid, n_inst).
    using WL = UnitLayout<WCAP, KW>;
    constexpr int W = WL::W;
    constexpr int NW = SkrLayout<PW>::WORDS;
    constexpr int HS = 2 * WCAP;  // hash slots (u16 each)
    constexpr int LOG_HS = WCAP == 512 ? 10 : 11;
    static_assert(WCAP == 512 || WCAP == 1024, "unit capacity");
    static_assert((1 << LOG_HS) == HS, "hash size");
    constexpr int NB_MAX = WL::NB_MAX, ECAP = WL::ECAP;
    extern __shared__ __align__(16) uint8_t smem3[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t h = warp % W, bar_id = 1 + warp / W;  // warp of the unit; named barrier of the pair (0 is __syncthreads')
    const uint32_t ul = h * 32 + lane;                    // lane inside the unit
    const bool first = ul == 0;                           // the unit's first lane: takes tickets, reports
    uint8_t *wb = smem3 + (size_t)(warp / W) * WL::BYTES;
    uint64_t *key0 = reinterpret_cast<uint64_t *>(wb);
    uint64_t *key1 = key0 + (KW == 2 ? WCAP : 0);
    uint16_t *tbl16 = reinterpret_cast<uint16_t *>(key0 + KW * WCAP);  // [2 * WCAP] hash slots: instance index + 1 of the group's leader
    uint32_t *cnt32 = reinterpret_cast<uint32_t *>(tbl16 + 2 * WCAP);  // [WCAP / 2] words = [WCAP] u16: instances per group, later the END of its id list
    uint16_t *cnt16 = reinterpret_cast<uint16_t *>(cnt32);
    uint32_t *cntlo32 = cnt32 + (W - 1) * WCAP / 2;                    // pair: [WCAP] u16 instances per group in the lower half (the counts
    uint16_t *cntlo16 = reinterpret_cast<uint16_t *>(cntlo32);         // of warp 0; cnt counts warp 1's, until the survivors pass adds them)
    uint16_t *grp = cnt16 + W * WCAP;                                  // [WCAP] leader (first inserted instance) of every instance's group
    uint16_t *rk = grp + WCAP;                                         // [WCAP] rank of the instance inside its group (pair: inside its half)
    uint8_t *eix = reinterpret_cast<uint8_t *>(rk + WCAP);             // [WCAP] entry of the instance (packed units)
    uint16_t *bstart = reinterpret_cast<uint16_t *>(eix + WCAP);       // [NB_MAX + 1] first instance of every bucket of the unit
    uint32_t *bmm = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(bstart) + WL::BSTART_BYTES);  // [NB_MAX] its m-mer code
    int32_t *eid = reinterpret_cast<int32_t *>(bmm + NB_MAX);          // [ECAP] read id of every entry
    uint8_t *ebk = reinterpret_cast<uint8_t *>(eid + ECAP);            // [ECAP] bucket ordinal of every entry
    PairXch xc{reinterpret_cast<uint32_t *>(ebk + ECAP), 0u};          // pair: exchange words
    // after the grouping the hash table is dead: its memory holds the survivor lists, then the unit's ids
    uint16_t *surv = tbl16;                               // [WCAP] instance index of every surviving leader, ascending
    uint16_t *sorted = surv + WCAP;                       // [WCAP] the same in table order (pair: first warp 1's survivors, see below)
    int32_t *idbuf = reinterpret_cast<int32_t *>(tbl16);  // [WCAP] the unit's ids in output order

    const int K = kl.K;
    const uint64_t kmask0 = (2 * K >= 64 * KW) ? ~0ull : ((1ull << (2 * K - 64 * (KW - 1))) - 1);
    const uint32_t unit_begin = chunk_bounds[chunk], unit_end = chunk_bounds[chunk + 1];
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t cls_mask = (uint32_t)(kl.nc - 1);
    // the ticket taken by the unit's first lane, to every lane of the unit (pair: the exchange's barrier also ends the unit)
    auto share_ticket = [&](uint32_t t) -> uint32_t {
        if (W == 1) return __shfl_sync(0xffffffffu, t, 0);
        return xc.put(h, lane, bar_id, __shfl_sync(0xffffffffu, t, 0))[0];
    };

    uint32_t u = 0;
    if (first) u = unit_begin + atomicAdd(&chunk_tickets[chunk], 1u);
    u = share_ticket(u);
    while (u < unit_end) {
        Unit3 un;
        {
            const uint32_t wv = lane < 8 ? reinterpret_cast<const uint32_t *>(units + u)[lane] : 0u;
            un.ent_begin = __shfl_sync(0xffffffffu, wv, 0);
            un.ent_end = __shfl_sync(0xffffffffu, wv, 1);
            un.n_inst = __shfl_sync(0xffffffffu, wv, 2);
            un.round = __shfl_sync(0xffffffffu, wv, 3);
            un.rounds = __shfl_sync(0xffffffffu, wv, 4);
            un.drange = __shfl_sync(0xffffffffu, wv, 5);
            un.ibase = __shfl_sync(0xffffffffu, wv, 6);
        }
        // the next ticket is taken now and read at the end of the unit (units do not depend on each other)
        uint32_t u_next = 0;
        if (first) u_next = unit_begin + atomicAdd(&chunk_tickets[chunk], 1u);
        const uint32_t u_cur = u;
        const bool is_round = un.rounds != 0;
        const uint32_t n_ent = un.ent_end - un.ent_begin;
        // packed: the unit's entries fit the per-entry tables and every instance remembers its entry; otherwise (a round of a split
        // atom, or one atom of very many entries) the unit is ONE bucket and the id pass walks the entries again
        const bool packed = !is_round && n_ent <= (uint32_t)ECAP;
        if (size_class) {
            const bool small = !is_round && un.n_inst <= G3_SMALL_INST && n_ent <= G3_SMALL_ENT;
            if (small != (size_class == 1u)) {  // the other launch's unit
                u = share_ticket(u_next);
                continue;
            }
        }
        if (is_round && un.n_inst == 0) {  // a round the cut did not need
            if (first) out.unit_out[u_cur] = UnitOut3{un.ibase, 0u, 0u, 0u};
            u = share_ticket(u_next);
            continue;
        }

        // ---- zero the hash table and the counters (contiguous)
        {
            uint4 *z = reinterpret_cast<uint4 *>(tbl16);
            for (uint32_t i = ul; i < (uint32_t)(WCAP * 4 + W * WCAP * 2) / 16; i += 32 * W) z[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        unit_sync<W>(bar_id);

        // ---- round units: the planner cut the atom's instances by ranges of d; mine is [dlo, dhi]
        int dlo = 0, dhi = 63;
        const uint32_t ibase = un.ibase;
        bool bad = false;
        if (is_round) {
            dlo = (int)(un.drange & 0xffu);
            dhi = (int)((un.drange >> 8) & 0xffu);
        }

        // ---- expansion: lane = entry.  Instance positions follow entry order (= key order, arrival order inside a key).
        uint32_t n_inst = 0, n_bkt = 0;
        if (!bad) {
            uint32_t carry_pos = 0, carry_ord = 0, prev_mm = 0xffffffffu;
            for (uint32_t e0 = 0; e0 < n_ent; e0 += 32 * W) {
                const uint32_t e = e0 + ul;
                uint32_t np = 0, t0 = 0, mm = 0xffffffffu, arrival = 0;
                bool rev = false;
                uint4 ha = make_uint4(0u, 0u, 0u, 0u), pa = ha, pb = ha;
                if (e < n_ent) {
                    const uint64_t en = ent[un.ent_begin + e];
                    const uint32_t slot = (uint32_t)en;
                    mm = (uint32_t)(en >> 32) >> kl.mshift;
                    const uint4 *rp = reinterpret_cast<const uint4 *>(skr + (uint64_t)(slot >> kl.cshift) * NW);
                    ha = rp[0];  // the whole record at once: header and payload
                    pa = rp[1];
                    if (PW == 4) pb = rp[2];
                    arrival = ha.x;
                    const uint32_t meta = ha.z;
                    rev = (meta >> 8) & 1u;
                    piece_of(meta, slot & cls_mask, kl, &t0, &np);
                    if (is_round && np) {  // windows with dlo <= so - t <= dhi
                        const int so = (int)((meta >> 16) & 0xffu);
                        int a = so - dhi, b = so - dlo;  // t in [a, b]
                        if (a < (int)t0) a = (int)t0;
                        if (b > (int)(t0 + np - 1)) b = (int)(t0 + np - 1);
                        if (dlo > dhi || b < a) np = 0;
                        else {
                            t0 = (uint32_t)a;
                            np = (uint32_t)(b - a + 1);
                        }
                    }
                }
                // buckets (runs of equal m-mer code) of the unit and instance positions
                uint32_t pm = __shfl_up_sync(0xffffffffu, mm, 1);
                if (lane == 0) {
                    if (W == 1) pm = prev_mm;
                    else pm = (e == 0 || e >= n_ent) ? 0xffffffffu : (uint32_t)(ent[un.ent_begin + e - 1] >> 32) >> kl.mshift;  // the entry before
                }
                const bool head = e < n_ent && mm != pm;
                uint32_t hs = warp_incl_scan_u32(head ? 1u : 0u, lane);
                uint32_t ps = warp_incl_scan_u32(np, lane);
                uint32_t hs_all = __shfl_sync(0xffffffffu, hs, 31), ps_all = __shfl_sync(0xffffffffu, ps, 31);
                if (W == 2) {  // 64-wide scans: warp 1's lanes follow warp 0's
                    const uint32_t *s = xc.put(h, lane, bar_id, hs_all, ps_all);
                    if (h) {
                        hs += s[0];
                        ps += s[1];
                    }
                    hs_all = s[0] + s[4];
                    ps_all = s[1] + s[5];
                }
                const uint32_t ord = carry_ord + hs - 1;  // bucket ordinal of this entry
                const uint32_t pos0 = carry_pos + ps - np;
                if (head && ord < (uint32_t)NB_MAX) {
                    bstart[ord] = (uint16_t)pos0;
                    bmm[ord] = mm;
                }
                carry_ord += hs_all;
                carry_pos += ps_all;
                if (W == 1) prev_mm = __shfl_sync(0xffffffffu, mm, 31);
                if (carry_pos > (uint32_t)WCAP || carry_ord > (uint32_t)NB_MAX || (!packed && carry_ord > 1u)) {  // cannot happen with the planner's bounds
                    bad = true;
                    break;
                }
                if (packed && e < n_ent) {
                    eid[e] = ids_by_arrival ? ids_by_arrival[arrival] : id_base + (int32_t)arrival;
                    ebk[e] = (uint8_t)ord;
                }
                if (np) {
                    Payload<PW> pl;
                    pl.set(pa, pb);
                    pl.skip(t0);
                    for (uint32_t i = 0; i < np; i++) {
                        uint64_t k0, k1;
                        front_kmer<PW, KW>(pl, K, rev, kmask0, &k0, &k1);
                        key0[pos0 + i] = k0;
                        if (KW == 2) key1[pos0 + i] = k1;
                        if (packed) eix[pos0 + i] = (uint8_t)e;
                        pl.advance(1);
                    }
                }
            }
            n_inst = carry_pos;
            n_bkt = carry_ord;
            if (!bad && first) bstart[n_bkt] = (uint16_t)n_inst;
        }
        unit_sync<W>(bar_id);
        if (bad) {  // give up on this unit: the batch is redone by another pipeline
            if (first) {
                atomicExch(&gc->overflow, 1u);
                out.unit_out[u_cur] = UnitOut3{ibase, 0u, 0u, 0u};
            }
            u = share_ticket(u_next);
            continue;
        }
        // my instance positions: [pbeg, pend).  Pair: warp 0 the lower half [0, mid), warp 1 the upper half [mid, n_inst).
        const uint32_t mid = W == 1 ? n_inst : min(n_inst, (n_inst + 63) / 64 * 32);
        const uint32_t pbeg = h ? mid : 0u, pend = h ? n_inst : mid;

        // ---- group: claim a slot with the instance index, compare keys through the instance arrays.  U instances per lane are in
        // flight together.  The rank of an instance inside its group follows position order: 32 positions per step, the peers of a
        // step are ranked by lane, the steps by the order in which their counter updates are issued.  A pair inserts into the same
        // table (the 16-bit CAS works across warps), but each warp counts its own half into its own counters (warp 0: cnt_lo,
        // warp 1: cnt), so the rank above is the rank inside the half.  Every position of the lower half precedes every position
        // of the upper half, so an instance's rank in position order = its rank inside its half, plus, in the upper half, the
        // group's count in the lower half (cnt_lo[leader], complete after the pair's barrier; the id pass adds it).  The result
        // does not depend on the timing of the two warps' atomics.
        uint32_t *cntw32 = (W == 2 && h == 0) ? cntlo32 : cnt32;
        for (uint32_t b0 = pbeg; b0 < pend; b0 += 32 * U) {
            uint64_t k0[U], k1[U];
            uint32_t lo[U], hi[U], idx[U], rep[U], cur[U];
            bool valid[U];
#pragma unroll
            for (int j = 0; j < U; j++) {
                const uint32_t p = b0 + j * 32 + lane;
                valid[j] = p < pend;
                k0[j] = valid[j] ? key0[p] : 0ull;
                k1[j] = (KW == 2 && valid[j]) ? key1[p] : 0ull;
                uint32_t o = 0;
                if (packed && valid[j]) o = ebk[eix[p]];
                lo[j] = bstart[o];  // instances of the same bucket: positions [lo, hi)
                hi[j] = bstart[o + 1];
                uint32_t hx = ((uint32_t)k0[j] * 0x9E3779B1u) ^ ((uint32_t)(k0[j] >> 32) * 0x85EBCA77u) ^ (o * 0xC2B2AE3Du);
                if (KW == 2) hx ^= ((uint32_t)k1[j] * 0x27D4EB2Fu) ^ ((uint32_t)(k1[j] >> 32) * 0x165667B1u);
                hx *= 0x9E3779B1u;
                idx[j] = hx >> (32 - LOG_HS);
                rep[j] = 0xffffffffu;
            }
#pragma unroll
            for (int j = 0; j < U; j++) cur[j] = valid[j] ? tbl16[idx[j]] : 0u;
#pragma unroll
            for (int j = 0; j < U; j++) {
                if (valid[j] && cur[j] == 0) {
                    const uint32_t p = b0 + j * 32 + lane;
                    const uint32_t old = atomicCAS(&tbl16[idx[j]], (unsigned short)0, (unsigned short)(p + 1));
                    if (old == 0) rep[j] = p;
                    else cur[j] = old;
                }
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                if (valid[j] && rep[j] == 0xffffffffu) {
                    const uint32_t r = cur[j] - 1;
                    if (r >= lo[j] && r < hi[j] && key0[r] == k0[j] && (KW == 1 || key1[r] == k1[j])) rep[j] = r;
                }
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                if (valid[j] && rep[j] == 0xffffffffu) {  // the slot holds another key: probe on
                    const uint32_t p = b0 + j * 32 + lane;
                    uint32_t ix = (idx[j] + 1) & (HS - 1);
                    for (;;) {
                        uint32_t c = tbl16[ix];
                        if (c == 0) {
                            c = atomicCAS(&tbl16[ix], (unsigned short)0, (unsigned short)(p + 1));
                            if (c == 0) {
                                rep[j] = p;
                                break;
                            }
                        }
                        const uint32_t r = c - 1;
                        if (r >= lo[j] && r < hi[j] && key0[r] == k0[j] && (KW == 1 || key1[r] == k1[j])) {
                            rep[j] = r;
                            break;
                        }
                        ix = (ix + 1) & (HS - 1);
                    }
                }
            }
            // ranks: all matches first, then all counter updates (issued in position order), then the broadcasts
            unsigned peers[U];
            uint32_t c[U];
#pragma unroll
            for (int j = 0; j < U; j++) peers[j] = __match_any_sync(0xffffffffu, valid[j] ? rep[j] : (0x10000u + lane));
#pragma unroll
            for (int j = 0; j < U; j++) {
                c[j] = 0;
                if (valid[j] && (int)lane == __ffs(peers[j]) - 1) {
                    const uint32_t sh = 16u * (rep[j] & 1u);
                    c[j] = (atomicAdd(&cntw32[rep[j] >> 1], (uint32_t)__popc(peers[j]) << sh) >> sh) & 0xffffu;
                }
                __syncwarp();  // the updates of step j must be issued before those of step j + 1 (diverged lanes could run ahead)
            }
#pragma unroll
            for (int j = 0; j < U; j++) {
                c[j] = __shfl_sync(0xffffffffu, c[j], __ffs(peers[j]) - 1);
                if (valid[j]) {
                    const uint32_t p = b0 + j * 32 + lane;
                    grp[p] = (uint16_t)rep[j];
                    rk[p] = (uint16_t)(c[j] + __popc(peers[j] & lt_mask));
                }
            }
        }
        unit_sync<W>(bar_id);

        // ---- leaders and survivors (keep iff count > cutoff, binning.c:1102); survivors are listed by ascending position.  Pair: a
        // group's count = cnt_lo + cnt, stored into cnt; warp 1 lists its survivors in `sorted` first and moves them behind warp 0's.
        uint32_t S = 0, N = 0, D = 0;
        uint16_t *my_surv = h ? sorted : surv;
        for (uint32_t b0 = pbeg; b0 < pend; b0 += 32 * U) {
            bool leader[U];
            uint32_t c[U];
#pragma unroll
            for (int j = 0; j < U; j++) {
                const uint32_t p = b0 + j * 32 + lane;
                leader[j] = p < pend && grp[p] == p;
            }
#pragma unroll
            for (int j = 0; j < U; j++) c[j] = leader[j] ? cnt16[b0 + j * 32 + lane] + (W == 2 ? cntlo16[b0 + j * 32 + lane] : 0u) : 0u;
#pragma unroll
            for (int j = 0; j < U; j++) {
                const uint32_t p = b0 + j * 32 + lane;
                const bool sv = leader[j] && (cutoff < 0 || c[j] > (uint32_t)cutoff);
                const unsigned lm = __ballot_sync(0xffffffffu, leader[j]), sm = __ballot_sync(0xffffffffu, sv);
                if (sv) {
                    my_surv[S + __popc(sm & lt_mask)] = (uint16_t)p;
                    if (W == 2) cnt16[p] = (uint16_t)c[j];
                } else if (leader[j]) cnt16[p] = 0xffffu;  // pruned
                S += __popc(sm);
                D += __popc(lm);
                N += sv ? c[j] : 0u;
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) N += __shfl_xor_sync(0xffffffffu, N, d);
        uint32_t S_lo = S;  // survivors of the lower half
        if (W == 2) {
            const uint32_t *s = xc.put(h, lane, bar_id, S, N, D);
            S_lo = s[0];
            S = s[0] + s[4];
            N = s[1] + s[5];
            D = s[2] + s[6];
        }
        const uint64_t kbase = ibase / out.kdiv;
        const bool oob = (uint64_t)ibase + N > out.id_cap || kbase + S > out.kmer_cap;  // cannot happen with the caller's bounds; never write out of range
        if (first) {
            out.unit_out[u_cur] = UnitOut3{ibase, oob ? 0u : S, oob ? 0u : N, 0u};
            atomicAdd(&gc->distinct, (unsigned long long)D);
            if (oob) atomicExch(&gc->overflow, 2u);
        }
        if (oob) {
            u = share_ticket(u_next);
            continue;
        }
        if (W == 2 && h) {
            __syncwarp();
            for (uint32_t x = lane; x < S - S_lo; x += 32) surv[S_lo + x] = sorted[x];
        }
        unit_sync<W>(bar_id);

        // ---- table order: buckets ascend with position already; inside a bucket every survivor counts the smaller keys
        for (uint32_t x0 = 0; x0 < S; x0 += 32 * W) {
            const uint32_t x = x0 + ul;
            if (x < S) {
                const uint32_t p = surv[x];
                uint32_t a = 0, a2 = S;
                if (n_bkt > 1) {
                    const uint32_t o = ebk[eix[p]];
                    const uint32_t blo = bstart[o], bhi = bstart[o + 1];
                    uint32_t b = S;  // first survivor with position >= blo
                    while (a < b) {
                        const uint32_t m = (a + b) >> 1;
                        if (surv[m] < blo) a = m + 1;
                        else b = m;
                    }
                    uint32_t b2 = S;  // first survivor with position >= bhi
                    a2 = a;
                    while (a2 < b2) {
                        const uint32_t m = (a2 + b2) >> 1;
                        if (surv[m] < bhi) a2 = m + 1;
                        else b2 = m;
                    }
                }
                const uint64_t k0 = key0[p], k1 = (KW == 2) ? key1[p] : 0ull;
                uint32_t rank = a;
                for (uint32_t t = a; t < a2; t++) {
                    const uint32_t q = surv[t];
                    const uint64_t q0 = key0[q];
                    bool less = q0 < k0;
                    if constexpr (KW == 2) less = less || (q0 == k0 && key1[q] < k1);
                    rank += less ? 1u : 0u;
                }
                sorted[rank] = (uint16_t)p;
            }
        }
        unit_sync<W>(bar_id);

        // ---- list offsets in table order: cnt[leader] becomes the END of its list inside the unit
        {
            uint32_t carry = 0;
            for (uint32_t x0 = 0; x0 < S; x0 += 32 * W) {
                const uint32_t x = x0 + ul;
                const uint32_t p = x < S ? sorted[x] : 0u;
                const uint32_t c = x < S ? cnt16[p] : 0u;
                uint32_t all;
                const uint32_t inc = unit_incl_scan<W>(c, lane, h, bar_id, xc, &all);
                if (x < S) cnt16[p] = (uint16_t)(carry + inc);
                carry += all;
            }
        }
        unit_sync<W>(bar_id);

        // ---- k-mers in table order, staged
        for (uint32_t x0 = 0; x0 < S; x0 += 32 * W) {
            const uint32_t x = x0 + ul;
            if (x < S) {
                const uint32_t p = sorted[x];
                const uint32_t beg = x ? cnt16[sorted[x - 1]] : 0u;
                const uint64_t g = kbase + x;
                out.codes[g * KW] = key0[p];
                if (KW == 2) out.codes[g * KW + 1] = key1[p];
                out.mmer[g] = bmm[n_bkt > 1 ? ebk[eix[p]] : 0u];
                out.loff[g] = beg;
            }
        }
        unit_sync<W>(bar_id);  // surv / sorted are dead from here on: the table's memory becomes the id buffer

        // ---- ids, newest first (binning.c:1059-1069): an instance's place = end of its list - 1 - its rank.  The unit's ids are
        // collected in shared memory and leave as one coalesced run.
        if (N) {
            if (packed) {
                for (uint32_t b0 = pbeg; b0 < pend; b0 += 32 * U) {
                    uint32_t end[U], r[U];
                    int32_t id[U];
#pragma unroll
                    for (int j = 0; j < U; j++) {
                        const uint32_t p = b0 + j * 32 + lane;
                        end[j] = 0xffffu;
                        r[j] = 0;
                        id[j] = 0;
                        if (p < pend) {
                            const uint32_t g = grp[p];
                            end[j] = cnt16[g];
                            r[j] = rk[p] + (W == 2 && h ? cntlo16[g] : 0u);
                            id[j] = eid[eix[p]];
                        }
                    }
#pragma unroll
                    for (int j = 0; j < U; j++)
                        if (end[j] != 0xffffu) idbuf[end[j] - 1u - r[j]] = id[j];
                }
            } else {  // lane = entry (the read id belongs to the record)
                uint32_t carry_pos = 0;
                for (uint32_t e0 = 0; e0 < n_ent; e0 += 32 * W) {
                    const uint32_t e = e0 + ul;
                    uint32_t np = 0, arrival = 0;
                    if (e < n_ent) {
                        const uint32_t slot = (uint32_t)ent[un.ent_begin + e];
                        const uint32_t *rec = skr + (uint64_t)(slot >> kl.cshift) * NW;
                        const uint32_t meta = rec[2];
                        arrival = rec[0];
                        uint32_t t0;
                        piece_of(meta, slot & cls_mask, kl, &t0, &np);
                        if (is_round && np) {
                            const int so = (int)((meta >> 16) & 0xffu);
                            int a = so - dhi, b = so - dlo;
                            if (a < (int)t0) a = (int)t0;
                            if (b > (int)(t0 + np - 1)) b = (int)(t0 + np - 1);
                            np = (dlo > dhi || b < a) ? 0u : (uint32_t)(b - a + 1);
                        }
                    }
                    uint32_t all;
                    const uint32_t ps = unit_incl_scan<W>(np, lane, h, bar_id, xc, &all);
                    const uint32_t pos0 = carry_pos + ps - np;
                    carry_pos += all;
                    if (np) {
                        const int32_t id = ids_by_arrival ? ids_by_arrival[arrival] : id_base + (int32_t)arrival;
                        for (uint32_t i = 0; i < np; i++) {
                            const uint32_t p = pos0 + i;
                            const uint32_t g = grp[p];
                            const uint32_t end = cnt16[g];
                            if (end != 0xffffu) idbuf[end - 1u - rk[p] - (W == 2 && p >= mid ? cntlo16[g] : 0u)] = id;
                        }
                    }
                }
            }
            unit_sync<W>(bar_id);
            int32_t *dst = out.ids + ibase;
            for (uint32_t i = ul; i < N; i += 32 * W) dst[i] = idbuf[i];
        }
        if (W == 1) __syncwarp();
        u = share_ticket(u_next);
    }
}

// ------------------------------------------------------------------ finalize: staging -> final place

struct UnitSN {  // {S << 32 | N} of the units of one chunk, 0 elsewhere
    const UnitOut3 *uo;
    const uint32_t *chunk_bounds;
    uint32_t chunk;
    __device__ __forceinline__ uint64_t operator()(uint64_t u) const {
        if (u < chunk_bounds[chunk] || u >= chunk_bounds[chunk + 1]) return 0ull;
        return ((uint64_t)uo[u].S << 32) | uo[u].N;
    }
};

// totals[c] = totals[c - 1] + what chunk c emitted, as {k-mers << 32 | ids} (totals[-1] = 0)
__global__ void v3_chunk_total_kernel(const uint64_t *__restrict__ chunk_sum, uint32_t chunk, unsigned long long *__restrict__ totals, G3Counters *__restrict__ gc,
                                      uint32_t n_chunks, int which) {
    const unsigned long long t = (chunk ? totals[chunk - 1] : 0ull) + *chunk_sum;
    totals[chunk] = t;
    if (chunk + 1 == n_chunks) {
        if (which == 0) {
            gc->total_kmers = t >> 32;
            gc->total_ids = t & 0xffffffffull;
        } else {
            gc->lsd_kmers = t >> 32;
            gc->lsd_ids = t & 0xffffffffull;
        }
    }
}

struct G3Final {  // this pass's part of the table (pointers at the pass's first k-mer / id)
    uint64_t *kmer_codes;   // [S * KW]
    uint32_t *kmer_mmer;    // [S]
    uint64_t *kmer_id_off;  // [S + 1]
    int32_t *read_ids;      // [N]
    uint64_t id_off_base;   // ids of the passes before this one (kmer_id_off holds offsets into the whole read_ids array)
};

// One warp per unit: copy its staged k-mers and ids to their place in the table (place = totals of all units before it).  The
// round units of a split atom are handled together by the warp that takes the atom's first round: the rounds are sorted runs of
// distinct k-mers, so a k-mer's place inside the atom = its index in its own run + the number of smaller k-mers in every other run.
// Long spans: every unit of the span appends its surviving k-mers to the arrays of the global sort, at a place given by a scan
// over the units of long spans (so a span's records are contiguous, spans in key order, and the sort by (m-mer, k-mer) permutes
// records only inside their span).  Indexed by the place p of a record BEFORE the sort: where its id list is staged and how long
// it is; indexed by a place q AFTER the sort: the k-mer's index in the table and what to add to the running list offset.
struct G3Lsd {
    const uint64_t *excl;  // [units] {k-mers << 32 | ids} of the long-span units before this one
    void *rec;             // Rec<KW> [n]
    uint32_t *src_off;     // [n] staging coordinate of the record's id list
    uint32_t *cnt;         // [n] its length
    uint32_t *fidx;        // [n] table index of the k-mer that ends up at this place
    uint32_t *nadj;        // [n] ids before the span that are not in long spans
    uint64_t cap;
};

struct UnitSNLong {  // {S << 32 | N} of the units of long spans of one chunk, 0 elsewhere
    const UnitOut3 *uo;
    const Unit3 *units;
    const uint32_t *chunk_bounds;
    uint32_t chunk;
    __device__ __forceinline__ uint64_t operator()(uint64_t u) const {
        if (u < chunk_bounds[chunk] || u >= chunk_bounds[chunk + 1]) return 0ull;
        const uint32_t sl = units[u].span_len;
        if (sl != SPAN_MEMBER_LONG && (sl <= SPAN_SHORT_MAX || sl == SPAN_MEMBER)) return 0ull;
        return ((uint64_t)uo[u].S << 32) | uo[u].N;
    }
};

// One warp per unit: copy its staged k-mers and ids to their place in the table (place = totals of all units before it).
// Short span: the warp of its first unit merges the units' runs — they hold distinct k-mers, each run ascending, so a k-mer's
// place inside the span = its index in its own run + the number of smaller k-mers in every other run.
template <int KW>
__device__ __forceinline__ void finalize3_unit(const Unit3 *__restrict__ units, const uint64_t *__restrict__ unit_excl, unsigned long long base,
                                               unsigned long long lsd_base, const G3Stage &st, const G3Final &fin, const G3Lsd &ls, G3Counters *gc, uint32_t u,
                                               uint32_t lane, bool only_long) {
    const uint32_t span_len = units[u].span_len;
    if (only_long && span_len != SPAN_MEMBER_LONG && (span_len <= SPAN_SHORT_MAX || span_len == SPAN_MEMBER)) return;  // done by the first run
    const uint64_t ex = unit_excl[u];
    const UnitOut3 uo = st.unit_out[u];
    const uint64_t Sb = (base >> 32) + (ex >> 32), Nb = (base & 0xffffffffull) + (ex & 0xffffffffull);
    if (span_len == 0) {
        // everything is loaded before anything is stored: one round trip to memory per batch of loads
        const uint64_t kb = uo.ibase / st.kdiv;
        for (uint32_t x0 = 0; x0 < uo.S; x0 += 128) {
            uint64_t c0[4], c1[4];
            uint32_t mm[4], lo[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t x = x0 + q * 32 + lane;
                if (x < uo.S) {
                    c0[q] = st.codes[(kb + x) * KW];
                    if (KW == 2) c1[q] = st.codes[(kb + x) * KW + 1];
                    mm[q] = st.mmer[kb + x];
                    lo[q] = st.loff[kb + x];
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t x = x0 + q * 32 + lane;
                if (x < uo.S) {
                    fin.kmer_codes[(Sb + x) * KW] = c0[q];
                    if (KW == 2) fin.kmer_codes[(Sb + x) * KW + 1] = c1[q];
                    fin.kmer_mmer[Sb + x] = mm[q];
                    fin.kmer_id_off[Sb + x] = fin.id_off_base + Nb + lo[q];
                }
            }
        }
        const int32_t *src = st.ids + uo.ibase;
        int32_t *dst = fin.read_ids + Nb;
        for (uint32_t i0 = 0; i0 < uo.N; i0 += 256) {
            int32_t v[8];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t i = i0 + q * 32 + lane;
                if (i < uo.N) v[q] = __ldcs(src + i);  // staged data is read once
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t i = i0 + q * 32 + lane;
                if (i < uo.N) dst[i] = v[q];
            }
        }
        return;
    }
    if (span_len == SPAN_MEMBER_LONG || (span_len > SPAN_SHORT_MAX && span_len != SPAN_MEMBER)) {
        // long span: hand this unit's k-mers to the global sort
        const uint64_t lx = ls.excl[u];
        const uint64_t q0 = (lsd_base >> 32) + (lx >> 32), nq0 = (lsd_base & 0xffffffffull) + (lx & 0xffffffffull);
        if (q0 + uo.S > ls.cap) {  // cannot happen with the caller's bounds
            if (lane == 0) atomicExch(&gc->overflow, 6u);
            return;
        }
        const uint64_t kb = uo.ibase / st.kdiv;
        Rec<KW> *rec = static_cast<Rec<KW> *>(ls.rec);
        for (uint32_t x = lane; x < uo.S; x += 32) {
            const uint64_t p = q0 + x;
            Rec<KW> r;
            r.k[0] = st.codes[(kb + x) * KW];
            if (KW == 2) r.k[KW - 1] = st.codes[(kb + x) * KW + 1];
            r.mmer = st.mmer[kb + x];
            r.arrival = (uint32_t)p;
            store_rec<KW>(rec + p, r);
            const uint32_t lo = st.loff[kb + x];
            ls.src_off[p] = uo.ibase + lo;
            ls.cnt[p] = (x + 1 < uo.S ? st.loff[kb + x + 1] : uo.N) - lo;
            ls.fidx[p] = (uint32_t)(Sb + x);
            ls.nadj[p] = (uint32_t)(Nb - nq0);
        }
        return;
    }
    // Short span (head or member): every unit's warp places its own run.  The runs of the span's units are ascending and hold
    // distinct k-mers, so a k-mer's place inside the span = its index in its own run + the number of smaller k-mers in every other
    // run, and its list starts after the lists of all those k-mers: own list offset + per other run the list offset of the first
    // k-mer that is not smaller (the staged list offsets of a unit ARE the prefix sums of its list lengths).  No unit waits for
    // another one and nothing staged is overwritten.
    uint32_t h = u;
    while (units[h].span_len == SPAN_MEMBER) h--;  // the span's first unit (at most SPAN_SHORT_MAX - 1 steps back)
    const uint32_t R = units[h].span_len;
    const uint64_t exh = unit_excl[h];
    const uint64_t Sh = (base >> 32) + (exh >> 32), Nh = (base & 0xffffffffull) + (exh & 0xffffffffull);
    if (uo.S == 0) return;
    const uint32_t j = u - h;
    const uint64_t kbj = uo.ibase / st.kdiv;
    const uint32_t mmer = st.mmer[kbj];  // every k-mer of the span has the same m-mer code
    for (uint32_t x0 = 0; x0 < uo.S; x0 += 32) {
        const uint32_t x = x0 + lane;
        uint32_t lo = 0, cnt = 0;
        uint64_t idoff = 0;
        if (x < uo.S) {
            const uint64_t k0 = st.codes[(kbj + x) * KW], k1 = KW == 2 ? st.codes[(kbj + x) * KW + 1] : 0ull;
            lo = st.loff[kbj + x];
            cnt = (x + 1 < uo.S ? st.loff[kbj + x + 1] : uo.N) - lo;
            uint32_t rank = x;
            idoff = lo;
            for (uint32_t j2 = 0; j2 < R; j2++) {
                if (j2 == j) continue;
                const UnitOut3 u2 = st.unit_out[h + j2];
                const uint64_t kb2 = u2.ibase / st.kdiv;
                uint32_t a = 0, b = u2.S;  // keys of run j2 smaller than mine
                while (a < b) {
                    const uint32_t m = (a + b) >> 1;
                    const uint64_t q0 = st.codes[(kb2 + m) * KW];
                    bool less = q0 < k0;
                    if constexpr (KW == 2) less = less || (q0 == k0 && st.codes[(kb2 + m) * KW + 1] < k1);
                    if (less) a = m + 1;
                    else b = m;
                }
                rank += a;
                idoff += a < u2.S ? st.loff[kb2 + a] : u2.N;
            }
            fin.kmer_codes[(Sh + rank) * KW] = k0;
            if (KW == 2) fin.kmer_codes[(Sh + rank) * KW + 1] = k1;
            fin.kmer_mmer[Sh + rank] = mmer;
            fin.kmer_id_off[Sh + rank] = fin.id_off_base + Nh + idoff;
        }
        const uint32_t nl = min(32u, uo.S - x0);
        for (uint32_t l0 = 0; l0 < nl; l0 += 4) {  // four lists per step, eight lanes each
            const uint32_t l = l0 + (lane >> 3);
            const uint32_t c = __shfl_sync(0xffffffffu, cnt, l & 31);
            const uint32_t so = __shfl_sync(0xffffffffu, lo, l & 31);
            const uint64_t d = __shfl_sync(0xffffffffu, idoff, l & 31);
            if (l < nl) {
                const int32_t *src = st.ids + uo.ibase + so;
                int32_t *dst = fin.read_ids + Nh + d;
                for (uint32_t i = lane & 7u; i < c; i += 8) dst[i] = src[i];
            }
        }
    }
}

template <int KW>
__global__ void __launch_bounds__(128, 12)
    finalize3_kernel(const Unit3 *__restrict__ units, const uint64_t *__restrict__ unit_excl, const unsigned long long *__restrict__ totals,
                     const unsigned long long *__restrict__ lsd_totals, G3Stage st, G3Final fin, G3Lsd ls, G3Counters *__restrict__ gc,
                     const uint32_t *__restrict__ chunk_bounds, uint32_t chunk, bool only_long) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t unit_begin = chunk_bounds[chunk], unit_end = chunk_bounds[chunk + 1];
    const unsigned long long base = chunk ? totals[chunk - 1] : 0ull;
    const unsigned long long lsd_base = chunk ? lsd_totals[chunk - 1] : 0ull;
    for (uint32_t u = unit_begin + blockIdx.x * 4 + (threadIdx.x >> 5); u < unit_end; u += gridDim.x * 4)
        finalize3_unit<KW>(units, unit_excl, base, lsd_base, st, fin, ls, gc, u, lane, only_long);
}

// ---- after the global sort of the long spans' k-mers (Rec<KW> sorted by (m-mer, k-mer); record.arrival = its place before the sort)
template <int KW>
struct LsdCnt {
    const Rec<KW> *rec;
    const uint32_t *cnt;
    __device__ __forceinline__ uint64_t operator()(uint64_t q) const { return cnt[rec[q].arrival]; }
};

template <int KW>
__global__ void lsd_place_kernel(const Rec<KW> *__restrict__ rec, uint64_t n, const uint64_t *__restrict__ dnew, G3Lsd ls, G3Final fin) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const Rec<KW> r = load_rec<KW>(rec + q);
    const uint64_t f = ls.fidx[q];
    fin.kmer_codes[f * KW] = r.k[0];
    if (KW == 2) fin.kmer_codes[f * KW + 1] = r.k[KW - 1];
    fin.kmer_mmer[f] = r.mmer;
    fin.kmer_id_off[f] = fin.id_off_base + dnew[q] + ls.nadj[q];
}

template <int KW>
__global__ void __launch_bounds__(256)
    lsd_lists_kernel(const Rec<KW> *__restrict__ rec, uint64_t n, const uint64_t *__restrict__ dnew, G3Lsd ls, const int32_t *__restrict__ stg_ids, G3Final fin) {
    const uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;  // eight lanes per list
    if (q >= n) return;
    const uint32_t p = rec[q].arrival;
    const uint32_t c = ls.cnt[p];
    const int32_t *src = stg_ids + ls.src_off[p];
    int32_t *dst = fin.read_ids + dnew[q] + ls.nadj[q];
    for (uint32_t i = threadIdx.x & 7u; i < c; i += 8) dst[i] = src[i];
}

// chunk_bounds[c] = first unit of chunk c, moved back to the first unit of a span so that no span straddles two chunks.
__global__ void v3_chunk_bounds_kernel(const Unit3 *__restrict__ units, const G3Counters *__restrict__ gc, uint32_t n_chunks, uint32_t *__restrict__ chunk_bounds) {
    const uint32_t nu = gc->n_units;
    for (uint32_t c = 0; c <= n_chunks; c++) {
        uint32_t b = (uint32_t)(((uint64_t)nu * c) / n_chunks);
        if (c == n_chunks) b = nu;
        else {
            while (b > 0 && b < nu && (units[b].span_len == SPAN_MEMBER || units[b].span_len == SPAN_MEMBER_LONG)) b--;  // back to the span's first unit
        }
        chunk_bounds[c] = b;
    }
}

// ------------------------------------------------------------------ host side

// cap: instances per unit, 512 or 1024 (gbin_set_tuning "v3_cap")
// Two grouping launches (see group3_kernel's size_class): for one-word k-mers at capacity 1024.
static bool v3_hybrid(const KeyLayout &kl, int cap_i) { return cap_i != 512 && kl.K <= 32; }
static Plan3 v3_plan_params(const KeyLayout &kl, int cap_i) {
    const uint32_t cap = cap_i == 512 ? 512u : 1024u;
    Plan3 pp{cap, cap / 8, cap / 4, (uint32_t)(kl.K - kl.M + 1), cap, cap / 8, cap / 4};  // NB_MAX and ECAP of UnitLayout
    if (v3_hybrid(kl, cap_i)) {
        pp.cap_s = G3_SMALL_INST;
        pp.nb_s = G3_SMALL_NB;
        pp.ecap_s = G3_SMALL_ENT;
    }
    return pp;
}

uint64_t v3_max_units(uint64_t n_inst, uint64_t n_runs, int cap) {
    const uint64_t c = cap == 512 ? 512 : 1024;
    // a packed unit holds at least one atom; an atom in rounds holds more than cap instances and gets at most 2 * ceil(instances / cap) + 1 units
    return n_runs + 5 * (n_inst / c) + 16;
}
size_t v3_unit_bytes() { return sizeof(Unit3); }
size_t v3_unit_out_bytes() { return sizeof(UnitOut3); }

struct PtrIn64 {
    const uint64_t *p;
    __device__ __forceinline__ uint64_t operator()(uint64_t j) const { return p[j]; }
};

// Units over the n_runs atoms.  nunits64 / base64: [n_runs + 1] u64 scratch each; atom3: [3 * n_runs] u32 scratch; spanlen: [n_runs] u32; head_run: [max_units].
int v3_plan_units(const uint16_t *sorted_info, const uint64_t *ent, const KeyLayout &kl, int cap, const uint32_t *inst_prefix, const uint32_t *run_start, uint64_t n_runs,
                  uint64_t *nunits64, uint64_t *base64, uint32_t *atom3, uint32_t *spanlen, uint32_t *head_run, void *scratch, void *units, uint64_t max_units,
                  void *gc_dev, uint32_t n_chunks, uint32_t *chunk_bounds, cudaStream_t st) {
    RunView3 rv{run_start, inst_prefix};
    const Plan3 pp = v3_plan_params(kl, cap);
    G3Counters *gc = static_cast<G3Counters *>(gc_dev);
    cudaMemsetAsync(gc, 0, sizeof(G3Counters), st);
    int l = 0;
    if (n_runs) {
        uint32_t *atom_c = atom3, *atom_e = atom3 + n_runs, *atom_mm = atom3 + 2 * n_runs;
        v3_atoms_kernel<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(rv, ent, n_runs, kl.mshift, atom_c, atom_e, atom_mm);
        const uint64_t walkers = (n_runs + PLAN_BLOCK - 1) / PLAN_BLOCK;
        v3_pack_kernel<<<(unsigned)((walkers + 127) / 128), 128, 0, st>>>(atom_c, atom_e, atom_mm, n_runs, pp, nunits64, spanlen);
        l += 2 + exclusive_scan<uint64_t, PtrIn64>(PtrIn64{nunits64}, base64, n_runs, static_cast<uint64_t *>(scratch), base64 + n_runs, st);
        v3_head_runs_kernel<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(nunits64, base64, n_runs, head_run);
        v3_fill_units_kernel<<<(unsigned)((max_units + 255) / 256), 256, 0, st>>>(rv, nunits64, spanlen, base64, base64 + n_runs, n_runs, head_run, static_cast<Unit3 *>(units), gc);
        v3_round_cuts_kernel<<<592, 128, 0, st>>>(sorted_info, static_cast<Unit3 *>(units), gc, pp.cap);
        l += 3;
    }
    v3_chunk_bounds_kernel<<<1, 1, 0, st>>>(static_cast<const Unit3 *>(units), gc, n_chunks, chunk_bounds);
    return l + 1;
}

// units in flight per CTA of the grouping kernel at capacity cap, and the CTA's threads (UnitLayout::W warps per unit)
static int v3_group_units(int cap) { return cap == 512 ? G3_WARPS : G3_PAIRS; }
static int v3_group_threads(int cap) { return v3_group_units(cap) * (cap == 512 ? UnitLayout<512, 1>::W : UnitLayout<1024, 1>::W) * 32; }

size_t v3_group_smem_bytes(int KW, int cap) {
    const size_t per_unit = cap == 512 ? (KW == 1 ? UnitLayout<512, 1>::BYTES : UnitLayout<512, 2>::BYTES)
                                       : (KW == 1 ? UnitLayout<1024, 1>::BYTES : UnitLayout<1024, 2>::BYTES);
    return per_unit * v3_group_units(cap);
}

int v3_group_launch(const void *skr, const uint64_t *ent, const void *units, const KeyLayout &kl, int cap, int cutoff, const int32_t *ids_by_arrival, int32_t id_base,
                    const V3Out &o, uint64_t max_units, uint64_t *unit_excl, uint64_t *lsd_excl, void *scan_scratch, void *gc_dev, const V3Chunks &ch, const V3Lsd &lsd,
                    bool finalize_only, int sm_count, KernelProf *prof, cudaStream_t st) {
    const int KW = kl.K <= 32 ? 1 : 2;
    const size_t smem = v3_group_smem_bytes(KW, cap);
    const int threads = v3_group_threads(cap), threads_s = v3_group_threads(512);
    cudaMemsetAsync(ch.tickets, 0, sizeof(uint32_t) * 2 * ch.n, st);
    const uint32_t kdiv = cutoff >= 0 ? (uint32_t)cutoff + 1u : 1u;
    G3Stage stg{o.stg_codes, o.stg_mmer, o.stg_loff, o.stg_ids, static_cast<UnitOut3 *>(o.unit_out), o.kmer_cap, o.id_cap, kdiv};
    G3Final fin{o.kmer_codes, o.kmer_mmer, o.kmer_id_off, o.read_ids, o.id_off_base};
    G3Lsd ls{lsd_excl, lsd.rec, lsd.src_off, lsd.cnt, lsd.fidx, lsd.nadj, lsd.cap};
    G3Counters *gc = static_cast<G3Counters *>(gc_dev);
    const uint32_t *sk = static_cast<const uint32_t *>(skr);
    const Unit3 *un = static_cast<const Unit3 *>(units);
    const int per_sm = g3_ctas_per_sm(smem);
    const bool hybrid = v3_hybrid(kl, cap);
    const size_t smem_s = v3_group_smem_bytes(KW, 512);
    const int per_sm_s = g3_ctas_per_sm(smem_s);
    int launches = 0;
    auto launch = [&](auto kern, auto kern_small, auto fin_kern) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (hybrid) cudaFuncSetAttribute(kern_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s);
        for (uint32_t c = 0; c < ch.n; c++) {
            if (!finalize_only) {
                bool on = prof && prof->begin(KK_SKR_GROUP, st);
                if (!hybrid) {
                    kern<<<sm_count * per_sm, threads, smem, st>>>(sk, ent, un, kl, cutoff, ids_by_arrival, id_base, stg, gc, ch.bounds, c, ch.tickets, 0u);
                } else {
                    // side by side: the large-unit kernel goes first with as many CTAs as its shared memory lets an SM hold, the
                    // small-unit kernel's CTAs take what is left of every SM and, being persistent, the room the other kernel leaves when
                    // it runs out of units (its tail is covered)
                    cudaEventRecord(ch.ev_fork, st);
                    cudaStreamWaitEvent(ch.aux, ch.ev_fork, 0);
                    kern<<<sm_count * per_sm, threads, smem, st>>>(sk, ent, un, kl, cutoff, ids_by_arrival, id_base, stg, gc, ch.bounds, c, ch.tickets, 2u);
                    kern_small<<<sm_count * per_sm_s, threads_s, smem_s, ch.aux>>>(sk, ent, un, kl, cutoff, ids_by_arrival, id_base, stg, gc, ch.bounds, c, ch.tickets + ch.n, 1u);
                    cudaEventRecord(ch.ev_join, ch.aux);
                    cudaStreamWaitEvent(st, ch.ev_join, 0);
                }
                if (prof) prof->end(on, hybrid ? 2 : 1, st);
                launches += hybrid ? 2 : 1;
            }
            bool on = prof && prof->begin(KK_V3_SPAN, st);
            int l = exclusive_scan<uint64_t, UnitSN>(UnitSN{stg.unit_out, ch.bounds, c}, unit_excl, max_units, static_cast<uint64_t *>(scan_scratch), ch.chunk_sum, st);
            v3_chunk_total_kernel<<<1, 1, 0, st>>>(ch.chunk_sum, c, ch.totals_dev, gc, ch.n, 0);
            l += exclusive_scan<uint64_t, UnitSNLong>(UnitSNLong{stg.unit_out, un, ch.bounds, c}, lsd_excl, max_units, static_cast<uint64_t *>(scan_scratch), ch.chunk_sum, st);
            v3_chunk_total_kernel<<<1, 1, 0, st>>>(ch.chunk_sum, c, ch.lsd_totals_dev, gc, ch.n, 1);
            // a second run (after the arrays of the global sort were allocated) only handles the long spans: the short-span merge is not idempotent
            fin_kern<<<sm_count * 12, 128, 0, st>>>(un, unit_excl, ch.totals_dev, ch.lsd_totals_dev, stg, fin, ls, gc, ch.bounds, c, finalize_only);
            if (prof) prof->end(on, l + 3, st);
            launches += l + 3;
            if (ch.totals_host) {
                cudaMemcpyAsync(ch.totals_host + c, ch.totals_dev + c, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
                cudaMemcpyAsync(ch.lsd_totals_host + c, ch.lsd_totals_dev + c, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
            }
            if (ch.done) cudaEventRecord(ch.done[c], st);
        }
    };
    // instances per lane in flight: 4 at capacity 1024, 2 at 512 (more warps per SM there: less need for instruction-level parallelism, smaller code)
    constexpr int W5 = G3_WARPS, P3 = G3_PAIRS;
    if (KW == 1) {
        if (cap == 512) launch(group3_kernel<2, 1, 512, W5, 2>, group3_kernel<2, 1, 512, W5, 2>, finalize3_kernel<1>);
        else launch(group3_kernel<2, 1, 1024, P3, 4>, group3_kernel<2, 1, 512, W5, 2>, finalize3_kernel<1>);
    } else {
        if (cap == 512) launch(group3_kernel<4, 2, 512, W5, 2>, group3_kernel<4, 2, 512, W5, 2>, finalize3_kernel<2>);
        else launch(group3_kernel<4, 2, 1024, P3, 4>, group3_kernel<4, 2, 512, W5, 2>, finalize3_kernel<2>);
    }
    return launches;
}

// ---- long spans, the common case: every span sorted on its own in shared memory.
// The records of a long span are contiguous, all carry the span's m-mer code, and consist of the ascending runs its units wrote
// (a unit's survivors are in k-mer order).  One CTA loads a span, finds the natural runs (a run ends where the k-mer decreases),
// and merges neighbouring runs pairwise, log2(runs) rounds between two buffers in shared memory: a k-mer's place in the merged
// run = its index in its own run + the number of smaller k-mers in the sibling run (binary search; k-mers of a span are
// distinct).  One read and one write of the records instead of the 11 radix passes of the global sort, which is kept for
// spans that do not fit shared memory (more than SS_CAP_BIG k-mers).
template <int KW>
struct RecHead {
    const Rec<KW> *rec;
    __device__ __forceinline__ uint32_t operator()(uint64_t p) const { return (p == 0 || rec[p].mmer != rec[p - 1].mmer) ? 1u : 0u; }
};
template <int KW>
__global__ void span_starts_kernel(const Rec<KW> *__restrict__ rec, uint64_t n, const uint32_t *__restrict__ idx, uint32_t *__restrict__ starts,
                                   uint32_t *__restrict__ n_spans, uint32_t *__restrict__ flag) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const bool head = p == 0 || rec[p].mmer != rec[p - 1].mmer;
    if (head) starts[idx[p]] = (uint32_t)p;
    if (p == n - 1) {
        const uint32_t total = idx[p] + (head ? 1u : 0u);  // idx = heads before p
        starts[total] = (uint32_t)n;
        *n_spans = total;
        *flag = 0u;
    }
}

constexpr int SS_RMAX = 1024;  // runs of a span (more: left to the global sort)
template <int KW, int CAP, int THREADS>
__global__ void __launch_bounds__(THREADS)
    span_sort_kernel(Rec<KW> *__restrict__ rec, const uint32_t *__restrict__ starts, const uint32_t *__restrict__ n_spans_ptr, uint32_t m_min, uint32_t m_max,
                     uint32_t *__restrict__ too_big) {
    extern __shared__ __align__(16) uint8_t ss_smem[];
    uint64_t *ka = reinterpret_cast<uint64_t *>(ss_smem);        // [KW][CAP] keys, buffer a
    uint64_t *kb = ka + KW * CAP;                                // buffer b
    uint16_t *sa = reinterpret_cast<uint16_t *>(kb + KW * CAP);  // [CAP] place of the record before the sort (relative to the span), buffer a
    uint16_t *sb = sa + CAP;
    uint16_t *ra = sb + CAP;  // [SS_RMAX + 2] run starts, buffer a
    uint16_t *rb = ra + SS_RMAX + 2;
    __shared__ uint32_t s_nruns;
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const uint32_t n_spans = *n_spans_ptr;
    for (uint32_t s = blockIdx.x; s < n_spans; s += gridDim.x) {
        const uint32_t b = starts[s], m = starts[s + 1] - b;
        if (m < m_min) continue;
        if (m > m_max) continue;  // another launch's span
        const uint32_t mmer = rec[b].mmer;
        for (uint32_t i = tid; i < m; i += THREADS) {
            const Rec<KW> r = load_rec<KW>(rec + b + i);
            ka[i] = r.k[0];
            if (KW == 2) ka[CAP + i] = r.k[KW - 1];
            sa[i] = (uint16_t)i;
        }
        __syncthreads();
        if (tid < 32) {  // natural runs
            uint32_t nr = 0;
            for (uint32_t i0 = 0; i0 < m; i0 += 32) {
                const uint32_t i = i0 + lane;
                bool head = false;
                if (i < m) {
                    head = i == 0 || ka[i] < ka[i - 1];
                    if (KW == 2 && i && ka[i] == ka[i - 1]) head = ka[CAP + i] < ka[CAP + i - 1];
                }
                const unsigned bal = __ballot_sync(0xffffffffu, head);
                if (head) {
                    const uint32_t pos = nr + __popc(bal & ((1u << lane) - 1u));
                    if (pos < (uint32_t)SS_RMAX) ra[pos] = (uint16_t)i;
                }
                nr += __popc(bal);
            }
            if (lane == 0) {
                s_nruns = nr;
                if (nr <= (uint32_t)SS_RMAX) ra[nr] = (uint16_t)m;
            }
        }
        __syncthreads();
        uint32_t nr = s_nruns;
        if (nr > (uint32_t)SS_RMAX) {
            if (tid == 0) atomicExch(too_big, 1u);
            __syncthreads();
            continue;
        }
        uint64_t *src_k = ka, *dst_k = kb;
        uint16_t *src_s = sa, *dst_s = sb, *src_r = ra, *dst_r = rb;
        while (nr > 1) {
            for (uint32_t i = tid; i < m; i += THREADS) {
                // my run: the last a with src_r[a] <= i
                uint32_t lo = 0, hi = nr;
                while (hi - lo > 1) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (src_r[mid] <= i) lo = mid;
                    else hi = mid;
                }
                const uint32_t a = lo, sib = a ^ 1u;
                const uint32_t pair0 = src_r[a & ~1u];
                uint32_t place;
                if (sib >= nr) {
                    place = i;  // the odd run out keeps its place
                } else {
                    const uint64_t k0 = src_k[i], k1 = KW == 2 ? src_k[CAP + i] : 0ull;
                    uint32_t l = src_r[sib], h = src_r[sib + 1];
                    const uint32_t sib0 = l;
                    while (l < h) {  // k-mers of the sibling run smaller than mine
                        const uint32_t mid = (l + h) >> 1;
                        const uint64_t q0 = src_k[mid];
                        bool less = q0 < k0;
                        if constexpr (KW == 2) less = less || (q0 == k0 && src_k[CAP + mid] < k1);
                        if (less) l = mid + 1;
                        else h = mid;
                    }
                    place = pair0 + (i - src_r[a]) + (l - sib0);
                }
                dst_k[place] = src_k[i];
                if (KW == 2) dst_k[CAP + place] = src_k[CAP + i];
                dst_s[place] = src_s[i];
            }
            const uint32_t nr2 = (nr + 1) >> 1;
            for (uint32_t a = tid; a <= nr2; a += THREADS) dst_r[a] = a < nr2 ? src_r[2 * a] : (uint16_t)m;
            __syncthreads();
            uint64_t *tk = src_k;
            src_k = dst_k;
            dst_k = tk;
            uint16_t *ts = src_s;
            src_s = dst_s;
            dst_s = ts;
            uint16_t *tr = src_r;
            src_r = dst_r;
            dst_r = tr;
            nr = nr2;
        }
        if (s_nruns > 1) {  // (one run: the span was in order already)
            for (uint32_t i = tid; i < m; i += THREADS) {
                Rec<KW> r;
                r.k[0] = src_k[i];
                if (KW == 2) r.k[KW - 1] = src_k[CAP + i];
                r.mmer = mmer;
                r.arrival = b + src_s[i];
                store_rec<KW>(rec + b + i, r);
            }
        }
        __syncthreads();
    }
}

// The same merge for a span that does not fit shared memory: the two buffers are the span's ranges of rec and rec2 in global
// memory (L2-resident: such a span is a few hundred KB), only the run starts live in shared memory.  One CTA per span.
constexpr int SS_RMAX_G = 8192;
template <int KW>
__device__ __forceinline__ bool rec_less(const Rec<KW> *a, uint64_t k0, uint64_t k1) {  // *a < (k0, k1), loads that bypass L1
    const uint64_t q0 = __ldcg(reinterpret_cast<const unsigned long long *>(&a->k[0]));
    if (KW == 1) return q0 < k0;
    if (q0 != k0) return q0 < k0;
    return __ldcg(reinterpret_cast<const unsigned long long *>(&a->k[KW - 1])) < k1;
}
template <int KW>
__global__ void __launch_bounds__(1024)
    span_sort_global_kernel(Rec<KW> *__restrict__ rec, Rec<KW> *__restrict__ rec2, const uint32_t *__restrict__ starts, const uint32_t *__restrict__ n_spans_ptr,
                            uint32_t m_min, uint32_t *__restrict__ too_big) {
    extern __shared__ __align__(16) uint8_t ssg_smem[];
    uint32_t *ra = reinterpret_cast<uint32_t *>(ssg_smem);  // [SS_RMAX_G + 2]
    uint32_t *rb = ra + SS_RMAX_G + 2;
    __shared__ uint32_t s_cnt[33];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t n_spans = *n_spans_ptr;
    for (uint32_t s = blockIdx.x; s < n_spans; s += gridDim.x) {
        const uint32_t b = starts[s], m = starts[s + 1] - b;
        if (m < m_min) continue;
        // natural runs: warp w takes the w-th 32nd of the span (count, prefix over the warps, list)
        const uint32_t per = (m + 31) / 32, c0 = warp * per, c1 = min(m, c0 + per);
        auto is_head = [&](uint32_t i) {
            if (i == 0) return true;
            const Rec<KW> *pr = rec + b + i - 1;
            const uint64_t k0 = __ldcg(reinterpret_cast<const unsigned long long *>(&rec[b + i].k[0]));
            const uint64_t k1 = KW == 2 ? __ldcg(reinterpret_cast<const unsigned long long *>(&rec[b + i].k[KW - 1])) : 0ull;
            return !rec_less<KW>(pr, k0, k1);  // the k-mer did not increase (k-mers of a span are distinct: it decreased)
        };
        uint32_t cnt = 0;
        for (uint32_t i0 = c0; i0 < c1; i0 += 32) {
            const uint32_t i = i0 + lane;
            cnt += __popc(__ballot_sync(0xffffffffu, i < c1 && is_head(i)));
        }
        if (lane == 0) s_cnt[warp] = cnt;
        __syncthreads();
        if (tid == 0) {
            uint32_t acc = 0;
            for (int w = 0; w < 32; w++) {
                const uint32_t c = s_cnt[w];
                s_cnt[w] = acc;
                acc += c;
            }
            s_cnt[32] = acc;
        }
        __syncthreads();
        uint32_t nr = s_cnt[32];
        if (nr > (uint32_t)SS_RMAX_G) {
            if (tid == 0) atomicExch(too_big, 1u);
            __syncthreads();
            continue;
        }
        {
            uint32_t at = s_cnt[warp];
            for (uint32_t i0 = c0; i0 < c1; i0 += 32) {
                const uint32_t i = i0 + lane;
                const bool head = i < c1 && is_head(i);
                const unsigned bal = __ballot_sync(0xffffffffu, head);
                if (head) ra[at + __popc(bal & ((1u << lane) - 1u))] = i;
                at += __popc(bal);
            }
            if (tid == 0) ra[nr] = m;
        }
        __syncthreads();
        Rec<KW> *src = rec + b, *dst = rec2 + b;
        uint32_t *src_r = ra, *dst_r = rb;
        const uint32_t nr0 = nr;
        while (nr > 1) {
            for (uint32_t i = tid; i < m; i += 1024) {
                uint32_t lo = 0, hi = nr;
                while (hi - lo > 1) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (src_r[mid] <= i) lo = mid;
                    else hi = mid;
                }
                const uint32_t a = lo, sib = a ^ 1u;
                Rec<KW> r;
                r.k[0] = __ldcg(reinterpret_cast<const unsigned long long *>(&src[i].k[0]));
                if (KW == 2) r.k[KW - 1] = __ldcg(reinterpret_cast<const unsigned long long *>(&src[i].k[KW - 1]));
                r.mmer = __ldcg(&src[i].mmer);
                r.arrival = __ldcg(&src[i].arrival);
                uint32_t place = i;
                if (sib < nr) {
                    uint32_t l = src_r[sib], h = src_r[sib + 1];
                    const uint32_t sib0 = l;
                    while (l < h) {
                        const uint32_t mid = (l + h) >> 1;
                        if (rec_less<KW>(src + mid, r.k[0], KW == 2 ? r.k[KW - 1] : 0ull)) l = mid + 1;
                        else h = mid;
                    }
                    place = src_r[a & ~1u] + (i - src_r[a]) + (l - sib0);
                }
                dst[place] = r;
            }
            const uint32_t nr2 = (nr + 1) >> 1;
            for (uint32_t a = tid; a <= nr2; a += 1024) dst_r[a] = a < nr2 ? src_r[2 * a] : m;
            __threadfence();
            __syncthreads();
            Rec<KW> *t = src;
            src = dst;
            dst = t;
            uint32_t *tr = src_r;
            src_r = dst_r;
            dst_r = tr;
            nr = nr2;
        }
        if (nr0 > 1 && src != rec + b) {  // an odd number of rounds: the result is in rec2
            for (uint32_t i = tid; i < m; i += 1024) {
                Rec<KW> r;
                r.k[0] = __ldcg(reinterpret_cast<const unsigned long long *>(&src[i].k[0]));
                if (KW == 2) r.k[KW - 1] = __ldcg(reinterpret_cast<const unsigned long long *>(&src[i].k[KW - 1]));
                r.mmer = __ldcg(&src[i].mmer);
                r.arrival = __ldcg(&src[i].arrival);
                rec[b + i] = r;
            }
        }
        __threadfence();
        __syncthreads();
    }
}

constexpr int SS_CAP_SMALL = 2048, SS_CAP_BIG = 8192;
template <int KW, int CAP>
constexpr size_t ss_smem_bytes() {
    return (size_t)2 * KW * CAP * 8 + (size_t)2 * CAP * 2 + (size_t)2 * (SS_RMAX + 2) * 2;
}

// Sorts every span of rec[0, n) (spans = runs of equal m-mer code) in shared memory.  work32: [2 n + 4] u32.  *too_big (device,
// = work32 + 2 n + 3) ends up non-zero when some span was left as it was.
template <int KW>
static int v3_span_sort(void *rec_v, void *rec2_v, uint64_t n, uint32_t *work32, void *scan_scratch, int sm_count, cudaStream_t st) {
    Rec<KW> *rec = static_cast<Rec<KW> *>(rec_v);
    uint32_t *idx = work32, *starts = work32 + n, *n_spans = work32 + 2 * n + 2, *flag = work32 + 2 * n + 3;
    int l = exclusive_scan<uint32_t, RecHead<KW>>(RecHead<KW>{rec}, idx, n, static_cast<uint32_t *>(scan_scratch), nullptr, st);
    span_starts_kernel<KW><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rec, n, idx, starts, n_spans, flag);
    constexpr int CS = SS_CAP_SMALL / KW, CB = SS_CAP_BIG / KW;
    constexpr size_t smem_s = ss_smem_bytes<KW, CS>(), smem_b = ss_smem_bytes<KW, CB>();
    cudaFuncSetAttribute(span_sort_kernel<KW, CS, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s);
    cudaFuncSetAttribute(span_sort_kernel<KW, CB, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b);
    const int per_sm = (int)((size_t)(227 * 1024) / (smem_s + 1024));
    span_sort_kernel<KW, CS, 256><<<sm_count * (per_sm < 1 ? 1 : per_sm), 256, smem_s, st>>>(rec, starts, n_spans, 2u, (uint32_t)CS, flag);
    span_sort_kernel<KW, CB, 1024><<<sm_count, 1024, smem_b, st>>>(rec, starts, n_spans, (uint32_t)CS + 1u, (uint32_t)CB, flag);
    constexpr size_t smem_g = (size_t)2 * (SS_RMAX_G + 2) * 4;
    cudaFuncSetAttribute(span_sort_global_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_g);
    span_sort_global_kernel<KW><<<sm_count * 2, 1024, smem_g, st>>>(rec, static_cast<Rec<KW> *>(rec2_v), starts, n_spans, (uint32_t)CB + 1u, flag);
    return l + 4;
}

// The long spans' k-mers (n records, appended by finalize3_kernel) are sorted by (m-mer, k-mer) — a permutation inside every span —
// and then written, with their id lists, to the table.  rec_a / rec_b: Rec<KW> [n] each; dnew: [n + 1] u64.
int v3_lsd_finish(const KeyLayout &kl, uint64_t n, void *rec_a, void *rec_b, void *radix_scratch, uint64_t *dnew, void *scan_scratch, const V3Out &o, const V3Lsd &lsd,
                  int sm_count, KernelProf *prof, cudaStream_t st) {
    if (n == 0) return 0;
    const int KW = kl.K <= 32 ? 1 : 2;
    bool in_b = false;
    int passes = 0;
    int l = 0;
    bool need_global = true;
    if (n < (1ull << 31)) {
        uint32_t *work32 = reinterpret_cast<uint32_t *>(dnew);  // [n + 2] u64 = [2 n + 4] u32; free until the list-length scan below
        bool on = prof && prof->begin(KK_V3_SPAN, st);
        const int ls_ = KW == 1 ? v3_span_sort<1>(rec_a, rec_b, n, work32, scan_scratch, sm_count, st) : v3_span_sort<2>(rec_a, rec_b, n, work32, scan_scratch, sm_count, st);
        if (prof) prof->end(on, ls_, st);
        l += ls_;
        uint32_t flag = 1;
        cudaMemcpyAsync(&flag, work32 + 2 * n + 3, sizeof flag, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) == cudaSuccess) need_global = flag != 0;
    }
    if (need_global) l += radix_sort_records(rec_a, rec_b, n, KW, kl.K, kl.M, radix_scratch, &in_b, &passes, prof, st);
    const void *sorted = in_b ? rec_b : rec_a;
    G3Final fin{o.kmer_codes, o.kmer_mmer, o.kmer_id_off, o.read_ids, o.id_off_base};
    G3Lsd ls{nullptr, nullptr, lsd.src_off, lsd.cnt, lsd.fidx, lsd.nadj, lsd.cap};
    bool on = prof && prof->begin(KK_V3_SPAN, st);
    int l2 = 0;
    if (KW == 1) {
        const Rec<1> *r = static_cast<const Rec<1> *>(sorted);
        l2 += exclusive_scan<uint64_t, LsdCnt<1>>(LsdCnt<1>{r, lsd.cnt}, dnew, n, static_cast<uint64_t *>(scan_scratch), nullptr, st);
        lsd_place_kernel<1><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(r, n, dnew, ls, fin);
        lsd_lists_kernel<1><<<(unsigned)((n * 8 + 255) / 256), 256, 0, st>>>(r, n, dnew, ls, o.stg_ids, fin);
    } else {
        const Rec<2> *r = static_cast<const Rec<2> *>(sorted);
        l2 += exclusive_scan<uint64_t, LsdCnt<2>>(LsdCnt<2>{r, lsd.cnt}, dnew, n, static_cast<uint64_t *>(scan_scratch), nullptr, st);
        lsd_place_kernel<2><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(r, n, dnew, ls, fin);
        lsd_lists_kernel<2><<<(unsigned)((n * 8 + 255) / 256), 256, 0, st>>>(r, n, dnew, ls, o.stg_ids, fin);
    }
    if (prof) prof->end(on, l2 + 2, st);
    return l + l2 + 2;
}

// ---- passes: a batch with more k-mer instances than 32-bit coordinates hold is grouped in several passes over consecutive
// ranges of the sorted entries, cut between m-mer buckets; every pass appends its part of the table.
constexpr uint32_t PASS_TILE = 1u << 16;
__global__ void pass_tile_sums_kernel(const uint16_t *__restrict__ info, uint64_t n_ent, unsigned long long *__restrict__ sums) {
    const uint64_t base = (uint64_t)blockIdx.x * PASS_TILE;
    unsigned long long acc = 0;
    for (uint64_t i = base + threadIdx.x; i < base + PASS_TILE && i < n_ent; i += blockDim.x) acc += info[i] & 0xffu;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    __shared__ unsigned long long s[8];
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += s[w];
        sums[blockIdx.x] = t;
    }
}
// bounds[i] (an entry index) is moved forward to the first entry of the next m-mer bucket; one thread per bound
__global__ void pass_bounds_kernel(const uint64_t *__restrict__ ent, uint64_t n_ent, int mshift, unsigned long long *__restrict__ bounds, uint32_t n_bounds) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bounds) return;
    unsigned long long b = bounds[i];
    if (b == 0 || b >= n_ent) return;
    const uint32_t mm = (uint32_t)(ent[b - 1] >> 32) >> mshift;
    while (b < n_ent && ((uint32_t)(ent[b] >> 32) >> mshift) == mm) b++;
    bounds[i] = b;
}
uint32_t v3_pass_tiles(uint64_t n_ent) { return (uint32_t)((n_ent + PASS_TILE - 1) / PASS_TILE); }
uint32_t v3_pass_tile_entries() { return PASS_TILE; }
int v3_pass_tile_sums(const uint16_t *sorted_info, uint64_t n_ent, unsigned long long *sums_dev, cudaStream_t st) {
    if (n_ent == 0) return 0;
    pass_tile_sums_kernel<<<v3_pass_tiles(n_ent), 256, 0, st>>>(sorted_info, n_ent, sums_dev);
    return 1;
}
int v3_pass_bounds(const uint64_t *ent, uint64_t n_ent, int mshift, unsigned long long *bounds_dev, uint32_t n_bounds, cudaStream_t st) {
    if (n_bounds == 0) return 0;
    pass_bounds_kernel<<<(n_bounds + 63) / 64, 64, 0, st>>>(ent, n_ent, mshift, bounds_dev, n_bounds);
    return 1;
}

// ---- how many different m-mer codes do the records hold?  (bitmap over the code space; decides the key layout)
__global__ void mmer_bitmap_kernel(const uint32_t *__restrict__ skr, int skr_words, uint64_t n_rec, uint32_t *__restrict__ bitmap) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rec) return;
    const uint32_t mm = skr[i * skr_words + 1];
    const uint32_t bit = 1u << (mm & 31u);
    if (!(bitmap[mm >> 5] & bit)) atomicOr(&bitmap[mm >> 5], bit);
}
__global__ void bitmap_count_kernel(const uint32_t *__restrict__ bitmap, uint64_t words, unsigned long long *__restrict__ count) {
    uint32_t c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (uint64_t)gridDim.x * blockDim.x) c += __popc(bitmap[i]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, (unsigned long long)c);
}
size_t v3_mmer_bitmap_bytes(int M) { return ((size_t)1 << (2 * M)) / 8 + 64; }
int v3_count_mmers(const void *skr, int skr_words, uint64_t n_rec, int M, uint32_t *bitmap, unsigned long long *count_dev, cudaStream_t st) {
    const uint64_t words = ((uint64_t)1 << (2 * M)) / 32;
    cudaMemsetAsync(bitmap, 0, words * 4, st);
    cudaMemsetAsync(count_dev, 0, sizeof(unsigned long long), st);
    if (n_rec == 0) return 0;
    mmer_bitmap_kernel<<<(unsigned)((n_rec + 255) / 256), 256, 0, st>>>(static_cast<const uint32_t *>(skr), skr_words, n_rec, bitmap);
    bitmap_count_kernel<<<592, 256, 0, st>>>(bitmap, words, count_dev);
    return 2;
}

}  // namespace gbin
