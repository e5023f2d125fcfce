// radix_sort.cu — stable LSD radix passes (8 bits per pass) over fixed-size records in HBM.
//
// Two users:
//   * pipeline v1: k-mer instance records Rec<KW> sorted on (mmer, kmer).  This replaces the reference's
//     per-k-mer hash chaining (zhash_get/zhash_set + strcmp along the chain, binning.c:1044-1058,
//     zhash.c:53-93): equal (m-mer, k-mer) keys become adjacent, and because every pass is stable and the
//     scan stage emits records in arrival order, the records of one key stay in arrival order — which is
//     what the linked list's head-insert order encodes (binning.c:1059-1069), read backwards;
//   * pipeline v2: super-k-mer records sorted on the m-mer code only (level 1 of the two-level store).
// With digit = owner_of_mmer(mmer, n_parts) the same pass is the stable owner partition of the multi-GPU path.
//
// Per pass: (1) per-tile digit histogram, (2) exclusive scan of the [256][tiles] table,
// (3) stable scatter: warp-level match ranking, tile-local reorder through shared memory so that
// every digit run leaves the SM as one contiguous, coalesced store.
#include "gbin_device.cuh"
#include "gbin_internal.h"
#include "lookback.cuh"
#include "prefix_scan.cuh"

namespace gbin {

constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_RADIX = 256;
#ifndef RS_ITEMS_32B
#define RS_ITEMS_32B 4
#endif

// A record seen as NU64 64-bit words (Rec<1>: 2, Rec<2>: 3, 32-byte super-k-mer: 4, 48-byte: 6).
template <int NU64>
struct __align__(8) Blob {
    uint64_t w[NU64];
};
template <int NU64>
__device__ __forceinline__ Blob<NU64> load_blob(const Blob<NU64> *p) {
    Blob<NU64> b;
    if (NU64 % 2 == 0) {  // 16-byte aligned record sizes: 128-bit accesses
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
#pragma unroll
        for (int i = 0; i < NU64 / 2; i++) {
            const uint4 v = q[i];
            b.w[2 * i] = (uint64_t)v.x | ((uint64_t)v.y << 32);
            b.w[2 * i + 1] = (uint64_t)v.z | ((uint64_t)v.w << 32);
        }
    } else {
#pragma unroll
        for (int i = 0; i < NU64; i++) b.w[i] = p->w[i];
    }
    return b;
}
template <int NU64>
__device__ __forceinline__ void store_blob(Blob<NU64> *p, const Blob<NU64> &b) {
    if (NU64 % 2 == 0) {
        uint4 *q = reinterpret_cast<uint4 *>(p);
#pragma unroll
        for (int i = 0; i < NU64 / 2; i++)
            q[i] = make_uint4((uint32_t)b.w[2 * i], (uint32_t)(b.w[2 * i] >> 32), (uint32_t)b.w[2 * i + 1], (uint32_t)(b.w[2 * i + 1] >> 32));
    } else {
#pragma unroll
        for (int i = 0; i < NU64; i++) p->w[i] = b.w[i];
    }
}

template <int NU64>
struct TileShape {  // records per thread: GBIN_RS_ITEMS_* below (payload registers per thread = 2 * NU64 * ITEMS)
    static constexpr int ITEMS = NU64 <= 2 ? 16 : (NU64 <= 4 ? RS_ITEMS_32B : 4);
    static constexpr int TILE = RS_THREADS * ITEMS;
};

struct DigitSel {
    int word64;    // which 64-bit word of the record holds the digit
    int shift;     // right shift inside that word
    uint32_t mod;  // 0: digit = (word >> shift) & 0xff ; else digit = owner_of_mmer((u32)(word >> shift), mod) (owner partition)
};

template <int NU64>
__device__ __forceinline__ uint32_t digit_of(const Blob<NU64> &r, const DigitSel &s) {
    uint64_t x = r.w[0];
#pragma unroll
    for (int i = 1; i < NU64; i++)
        if (s.word64 == i) x = r.w[i];  // no dynamic indexing: keeps records in registers
    x >>= s.shift;
    return s.mod ? owner_of_mmer((uint32_t)x, s.mod) : (uint32_t)x & 0xffu;
}

// DROP: records whose key (high half of word 0) is all ones are left out (the empty pieces of the entry sort); n_dev: the
// record count is read from device memory (what is left after the pass that dropped them).
template <int NU64, bool DROP>
__global__ void __launch_bounds__(RS_THREADS)
    radix_hist_kernel(const Blob<NU64> *__restrict__ in, uint64_t n, DigitSel sel, uint32_t *__restrict__ tile_hist, uint32_t ntiles,
                      const unsigned long long *__restrict__ n_dev) {
    constexpr bool drop_ones = DROP;
    constexpr int ITEMS = TileShape<NU64>::ITEMS, TILE = TileShape<NU64>::TILE;
    __shared__ uint32_t h[RS_RADIX];
    h[threadIdx.x] = 0;
    __syncthreads();
    if (n_dev) n = *n_dev;  // the record count is only known on the device (entries left after the pass that dropped the empty ones)
    const uint64_t base = (uint64_t)blockIdx.x * TILE;
#pragma unroll 4
    for (int i = 0; i < ITEMS; i++) {
        const uint64_t j = base + (uint64_t)i * RS_THREADS + threadIdx.x;
        if (j < n) {
            const Blob<NU64> r = load_blob<NU64>(in + j);
            if (!(drop_ones && (uint32_t)(r.w[0] >> 32) == 0xffffffffu)) atomicAdd(&h[digit_of<NU64>(r, sel)], 1u);
        }
    }
    __syncthreads();
    tile_hist[(uint64_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

template <int NU64, bool DROP>
__global__ void __launch_bounds__(RS_THREADS)
    radix_scatter_kernel(const Blob<NU64> *__restrict__ in, Blob<NU64> *__restrict__ out, uint64_t n, DigitSel sel,
                         const uint32_t *__restrict__ tile_off, uint32_t ntiles, char *const *__restrict__ dst_tab, uint64_t *__restrict__ side,
                         const uint16_t *__restrict__ slot_info, uint16_t *__restrict__ sorted_info, const unsigned long long *__restrict__ n_dev) {
    constexpr bool drop_ones = DROP;
    constexpr int ITEMS = TileShape<NU64>::ITEMS, TILE = TileShape<NU64>::TILE;
    if (n_dev) n = *n_dev;
    if ((uint64_t)blockIdx.x * TILE >= n) return;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    Blob<NU64> *exch = reinterpret_cast<Blob<NU64> *>(smem_raw);
    uint32_t *wc = reinterpret_cast<uint32_t *>(smem_raw + (size_t)TILE * sizeof(Blob<NU64>));  // [RS_WARPS][256]
    uint32_t *dstart = wc + RS_WARPS * RS_RADIX;
    uint32_t *goff = dstart + RS_RADIX;
    // Owner exchange (dst_tab != nullptr, digit = owner < XCHG_MAX_WORLD): digit d's run goes to dst_tab[d], the owner's
    // receive buffer (peer memory over NVLink) already offset so that the run lands behind the lower ranks' records.
    __shared__ char *s_dst[XCHG_MAX_WORLD];
    if (dst_tab && threadIdx.x < XCHG_MAX_WORLD) s_dst[threadIdx.x] = dst_tab[threadIdx.x];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t base = (uint64_t)blockIdx.x * TILE;
    const uint32_t count = (uint32_t)min((uint64_t)TILE, n - base);  // records of the tile; `kept` of them are scattered (drop_ones: entries with the all-ones key are left out)
    for (uint32_t i = tid; i < RS_WARPS * RS_RADIX; i += RS_THREADS) wc[i] = 0;
    __syncthreads();

    // warp `warp` owns the contiguous slice [warp*32*ITEMS, (warp+1)*32*ITEMS) of the tile, ITEMS rounds of 32
    Blob<NU64> items[ITEMS];
    uint32_t rank[ITEMS];
    uint32_t *mywc = wc + warp * RS_RADIX;
    const uint32_t lt_mask = (1u << lane) - 1;
    // all loads of the thread are issued before anything waits for one of them (a load per ranking round would put a round trip to
    // memory on the critical path of every round)
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
        const uint32_t idx = warp * (32 * ITEMS) + r * 32 + lane;
        if (idx < count) items[r] = load_blob<NU64>(in + base + idx);
    }
    uint32_t keep_mask = 0;  // bit r: this thread's record of round r takes part
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
        const uint32_t idx = warp * (32 * ITEMS) + r * 32 + lane;
        const bool valid = idx < count && !(drop_ones && (uint32_t)(items[r].w[0] >> 32) == 0xffffffffu);
        keep_mask |= valid ? (1u << r) : 0u;
        const unsigned act = __ballot_sync(0xffffffffu, valid);
        rank[r] = 0;
        if (valid) {
            const uint32_t d = digit_of<NU64>(items[r], sel);
            // lanes with my digit: eight ballots (one per bit) — a fixed cost, whereas MATCH.ANY iterates over the distinct values in the warp
            unsigned peers = act;
#pragma unroll
            for (int b = 0; b < 8; b++) {
                const bool bit = (d >> b) & 1u;
                const unsigned m = __ballot_sync(act, bit);
                peers &= bit ? m : ~m;
            }
            const int leader = __ffs(peers) - 1;
            uint32_t c = 0;
            if ((int)lane == leader) {
                c = mywc[d];
                mywc[d] = c + __popc(peers);
            }
            c = __shfl_sync(peers, c, leader);
            rank[r] = c + __popc(peers & lt_mask);
        }
        __syncwarp();
    }
    __syncthreads();
    uint32_t kept;  // records of the tile that are scattered: all of them unless drop_ones
    {  // thread = digit: exclusive scan over warps, then over digits
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) {
            const uint32_t t = wc[w * RS_RADIX + tid];
            wc[w * RS_RADIX + tid] = run;
            run += t;
        }
        uint32_t tot;
        const uint32_t excl = block_exclusive_scan<uint32_t>(run, &tot);
        kept = drop_ones ? tot : count;
        dstart[tid] = excl;
        goff[tid] = tile_off[(uint64_t)tid * ntiles + blockIdx.x] - excl;  // mod 2^32, n < 2^32
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ITEMS; r++) {
        if ((keep_mask >> r) & 1u) {
            const uint32_t d = digit_of<NU64>(items[r], sel);
            exch[dstart[d] + mywc[d] + rank[r]] = items[r];
        }
    }
    __syncthreads();
    if (dst_tab) {
        for (uint32_t i = tid; i < kept; i += RS_THREADS) {
            const Blob<NU64> r = exch[i];
            const uint32_t d = digit_of<NU64>(r, sel);
            char *bp = s_dst[d];
            if (bp) store_blob<NU64>(reinterpret_cast<Blob<NU64> *>(bp) + (uint32_t)(goff[d] + i), r);
        }
        return;
    }
    for (uint32_t i = tid; i < kept; i += RS_THREADS) {
        const Blob<NU64> r = exch[i];
        const uint32_t d = digit_of<NU64>(r, sel);
        const uint32_t pos = (uint32_t)(goff[d] + i);
        store_blob<NU64>(out + pos, r);
        // last pass of the super-k-mer sort: {m-mer code, windows} of every record in sorted order, 8 bytes instead of the
        // whole record for the planning scans that follow
        if constexpr (NU64 >= 2) {
            if (side) side[pos] = (r.w[0] & 0xffffffff00000000ull) | (r.w[1] & 0xffull);
        } else {
            // last pass of the entry sort: what the planner needs of every piece (windows, smallest d), in sorted order
            if (sorted_info) sorted_info[pos] = slot_info[(uint32_t)r.w[0]];
        }
    }
}

// ------------------------------------------------------------------ owner exchange over peer memory
// One process per GPU; every rank maps every peer's receive buffer and XchgShared block (CUDA IPC, set up once by
// capi.cu).  Per exchange (all on the rank's stream, no host round trip and no NCCL call):
//   1. the usual per-tile histogram of digit = owner_of_mmer(mmer, world) and its scan (above);
//   2. xchg_counts_kernel: this rank's per-owner counts go into row `rank` of every peer's count matrix, a flag with the
//      exchange's epoch follows (release at system scope); the kernel then waits for every rank's row, derives where its
//      records start inside each owner's buffer (behind the records of the lower ranks: arrival order is kept) and how
//      many records it will receive itself;
//   3. the scatter kernel stores every owner's run straight into that owner's buffer (NVLink peer stores);
//   4. xchg_done_kernel: "my stores are done" to every peer, then waits for all peers' flags: the receive buffer is
//      complete.  A rank publishes the counts of its NEXT exchange only after it has consumed its receive buffer (stream
//      order), so waiting for all rows in step 2 also means every receive buffer is free again.
// Waits are bounded (XchgPlan::timeout_cycles, two minutes unless set) so a missing peer yields an error code, not a hung GPU.

__device__ __forceinline__ void st_release_sys(unsigned int *p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
constexpr long long XCHG_TIMEOUT_CYCLES = 240000000000ll;  // about 2 minutes (gbin_set_tuning "xchg_timeout_ms" sets XchgPlan::timeout_cycles)

__device__ __forceinline__ bool xchg_wait_flag(const unsigned int *p, unsigned int epoch, long long timeout_cycles) {
    const long long t0 = clock64();
    const long long limit = timeout_cycles > 0 ? timeout_cycles : XCHG_TIMEOUT_CYCLES;
    while (ld_acquire_sys(p) != epoch) {
        if (clock64() - t0 > limit) return false;
        __nanosleep(200);
    }
    return true;
}

__global__ void xchg_counts_kernel(const uint32_t *__restrict__ tile_off, uint32_t ntiles, uint64_t n, XchgPlan xp, uint32_t rec_bytes) {
    const uint32_t lane = threadIdx.x, G = xp.world, me = xp.rank;
    unsigned long long cnt = 0, start = 0;
    if (lane < G) {
        start = n ? tile_off[(uint64_t)lane * ntiles] : 0;
        const unsigned long long end = n ? ((lane + 1 < RS_RADIX) ? tile_off[(uint64_t)(lane + 1) * ntiles] : n) : 0;
        cnt = end - start;
        for (uint32_t p = 0; p < G; p++) xp.peer_sh[p]->counts[me * XCHG_MAX_WORLD + lane] = cnt;
    }
    __threadfence_system();
    __syncwarp();
    bool ok = true;
    if (lane < G) {
        st_release_sys(&xp.peer_sh[lane]->count_flag[me], xp.epoch);
        ok = xchg_wait_flag(&xp.peer_sh[me]->count_flag[lane], xp.epoch, xp.timeout_cycles);
    }
    const bool all_here = __all_sync(0xffffffffu, ok);
    unsigned long long off = 0, tot = 0;
    if (all_here && lane < G) {
        for (uint32_t s = 0; s < G; s++) {
            const unsigned long long c = ld_relaxed_sys_u64(&xp.peer_sh[me]->counts[s * XCHG_MAX_WORLD + lane]);
            if (s < me) off += c;
            tot += c;
        }
        ok = tot <= xp.cap[lane];
    }
    const bool fits = __all_sync(0xffffffffu, ok);
    const unsigned long long n_in = __shfl_sync(0xffffffffu, tot, me);
    if (lane < XCHG_MAX_WORLD)
        xp.dst_tab[lane] = (all_here && fits && lane < G)
                               ? reinterpret_cast<char *>(xp.peer_recv[lane]) + ((long long)off - (long long)start) * (long long)rec_bytes
                               : nullptr;
    if (lane < G) xp.result->sent[lane] = cnt;
    if (lane == 0) {
        xp.result->n_in = n_in;
        xp.result->status = !all_here ? 2u : (fits ? 0u : 1u);
    }
}

__global__ void xchg_done_kernel(XchgPlan xp) {
    const uint32_t lane = threadIdx.x, G = xp.world, me = xp.rank;
    __threadfence_system();
    bool ok = true;
    if (lane < G) {
        st_release_sys(&xp.peer_sh[lane]->done_flag[me], xp.epoch);
        ok = xchg_wait_flag(&xp.peer_sh[me]->done_flag[lane], xp.epoch, xp.timeout_cycles);
    }
    if (!__all_sync(0xffffffffu, ok) && lane == 0) xp.result->status = 2u;
}

__global__ void part_counts_kernel(const uint32_t *__restrict__ tile_off, uint32_t ntiles, uint32_t nparts, uint64_t n,
                                   uint64_t *__restrict__ counts) {
    const uint32_t p = threadIdx.x;
    if (p >= nparts) return;
    const uint64_t lo = tile_off[(uint64_t)p * ntiles];
    const uint64_t hi = (p + 1 < RS_RADIX) ? tile_off[(uint64_t)(p + 1) * ntiles] : n;
    counts[p] = hi - lo;
}

static inline uint32_t ntiles_of(uint64_t n, int tile) { return (uint32_t)((n + tile - 1) / tile); }

static uint32_t ntiles_any(int nu64, uint64_t n) {
    switch (nu64) {
        case 1: return ntiles_of(n, TileShape<1>::TILE);
        case 2: return ntiles_of(n, TileShape<2>::TILE);
        case 3: return ntiles_of(n, TileShape<3>::TILE);
        case 4: return ntiles_of(n, TileShape<4>::TILE);
        default: return ntiles_of(n, TileShape<6>::TILE);
    }
}

size_t radix_scratch_bytes(uint64_t n) {
    const uint64_t table = (uint64_t)RS_RADIX * ntiles_of(n ? n : 1, TileShape<6>::TILE);  // smallest tile of any record size
    return (table + scan_scratch_elems(table) + 16) * sizeof(uint32_t);
}

template <int NU64>
static int one_pass(const void *in_v, void *out_v, uint64_t n, const DigitSel &sel, uint32_t *scratch, KernelProf *prof, cudaStream_t st,
                    const XchgPlan *xp = nullptr, uint64_t *side = nullptr, const uint16_t *slot_info = nullptr, uint16_t *sorted_info = nullptr,
                    const unsigned long long *n_dev = nullptr, bool drop_ones = false) {
    const Blob<NU64> *in = static_cast<const Blob<NU64> *>(in_v);
    Blob<NU64> *out = static_cast<Blob<NU64> *>(out_v);
    constexpr int TILE = TileShape<NU64>::TILE;
    if (n == 0) {
        if (!xp) return 0;
        // nothing to send: still take part in the count exchange and the completion barrier
        xchg_counts_kernel<<<1, 32, 0, st>>>(scratch, 0, 0, *xp, (uint32_t)sizeof(Blob<NU64>));
        xchg_done_kernel<<<1, 32, 0, st>>>(*xp);
        return 2;
    }
    const uint32_t nt = ntiles_of(n, TILE);
    const uint64_t table = (uint64_t)RS_RADIX * nt;
    uint32_t *tile_hist = scratch;
    uint32_t *scan_tmp = scratch + table;
    int launches = 0;
    bool on = prof && prof->begin(KK_RADIX_HIST, st);
    if (NU64 == 1 && drop_ones) radix_hist_kernel<NU64, NU64 == 1><<<nt, RS_THREADS, 0, st>>>(in, n, sel, tile_hist, nt, n_dev);
    else radix_hist_kernel<NU64, false><<<nt, RS_THREADS, 0, st>>>(in, n, sel, tile_hist, nt, n_dev);
    if (prof) prof->end(on, 1, st);
    launches++;
    on = prof && prof->begin(KK_RADIX_TILESCAN, st);
    const int ls = exclusive_scan<uint32_t, PtrIn<uint32_t>>(PtrIn<uint32_t>{tile_hist}, tile_hist, table, scan_tmp, nullptr, st);
    if (prof) prof->end(on, ls, st);
    launches += ls;
    const size_t smem = (size_t)TILE * sizeof(Blob<NU64>) + (RS_WARPS * RS_RADIX + 2 * RS_RADIX) * sizeof(uint32_t);
    cudaFuncSetAttribute(radix_scatter_kernel<NU64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (NU64 == 1) cudaFuncSetAttribute(radix_scatter_kernel<NU64, NU64 == 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    on = prof && prof->begin(KK_RADIX_SCATTER, st);
    if (xp) {  // counts to every peer, wait for theirs, per-owner destinations
        xchg_counts_kernel<<<1, 32, 0, st>>>(tile_hist, nt, n, *xp, (uint32_t)sizeof(Blob<NU64>));
        launches++;
    }
    if (NU64 == 1 && drop_ones)
        radix_scatter_kernel<NU64, NU64 == 1><<<nt, RS_THREADS, smem, st>>>(in, out, n, sel, tile_hist, nt, xp ? xp->dst_tab : nullptr, side, slot_info, sorted_info, n_dev);
    else
        radix_scatter_kernel<NU64, false><<<nt, RS_THREADS, smem, st>>>(in, out, n, sel, tile_hist, nt, xp ? xp->dst_tab : nullptr, side, slot_info, sorted_info, n_dev);
    if (prof) prof->end(on, 1, st);
    if (xp) {
        xchg_done_kernel<<<1, 32, 0, st>>>(*xp);
        launches++;
    }
    return launches + 1;
}

static int one_pass_any(int nu64, const void *in, void *out, uint64_t n, const DigitSel &sel, uint32_t *scratch, KernelProf *prof,
                        cudaStream_t st, const XchgPlan *xp = nullptr, uint64_t *side = nullptr, const uint16_t *slot_info = nullptr,
                        uint16_t *sorted_info = nullptr, const unsigned long long *n_dev = nullptr, bool drop_ones = false) {
    switch (nu64) {
        case 1: return one_pass<1>(in, out, n, sel, scratch, prof, st, xp, side, slot_info, sorted_info, n_dev, drop_ones);
        case 2: return one_pass<2>(in, out, n, sel, scratch, prof, st, xp, side);
        case 3: return one_pass<3>(in, out, n, sel, scratch, prof, st, xp, side);
        case 4: return one_pass<4>(in, out, n, sel, scratch, prof, st, xp, side);
        default: return one_pass<6>(in, out, n, sel, scratch, prof, st, xp, side);
    }
}

// v1: instance records {u64 k[KW]; u32 mmer; u32 arrival}: k-mer words are w[0..KW-1] (most significant first),
// the m-mer code is the low half of w[KW].
int radix_sort_records(void *a, void *b, uint64_t n, int KW, int K, int M, void *scratch, bool *result_in_b, int *passes_out,
                       KernelProf *prof, cudaStream_t st) {
    *result_in_b = false;
    *passes_out = 0;
    if (n == 0) return 0;
    int launches = 0, passes = 0;
    void *src = a, *dst = b;
    auto run = [&](DigitSel sel) {
        launches += one_pass_any(KW + 1, src, dst, n, sel, static_cast<uint32_t *>(scratch), prof, st);
        void *t = src;
        src = dst;
        dst = t;
        passes++;
    };
    // least significant digits first: k-mer low word ... k-mer high word, then the m-mer code
    int kbits = 2 * K;
    for (int w = KW - 1; w >= 0; w--) {
        const int bits = kbits > 64 ? 64 : kbits;
        for (int s = 0; s < bits; s += 8) run(DigitSel{w, s, 0});
        kbits -= bits;
    }
    for (int s = 0; s < 2 * M; s += 8) run(DigitSel{KW, s, 0});
    *result_in_b = (src == b);
    *passes_out = passes;
    return launches;
}

int radix_partition_by_owner(const void *in, void *out, uint64_t n, int KW, uint32_t n_parts, void *scratch, uint64_t *d_counts,
                             cudaStream_t st) {
    if (n == 0) {
        cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * n_parts, st);
        return 0;
    }
    const DigitSel sel{KW, 0, n_parts};
    const int launches = one_pass_any(KW + 1, in, out, n, sel, static_cast<uint32_t *>(scratch), nullptr, st);
    part_counts_kernel<<<1, RS_RADIX, 0, st>>>(static_cast<uint32_t *>(scratch), ntiles_any(KW + 1, n), n_parts, n, d_counts);
    return launches + 1;
}

// v2: super-k-mer records (skr.cuh): word 1 (= high half of w[0]) is the m-mer code.
int radix_sort_skr_by_mmer(void *a, void *b, uint64_t n, int skr_words, int M, void *scratch, bool *result_in_b, int *passes_out,
                           uint64_t *side_out, KernelProf *prof, cudaStream_t st) {
    *result_in_b = false;
    *passes_out = 0;
    if (n == 0) return 0;
    int launches = 0, passes = 0;
    void *src = a, *dst = b;
    for (int s = 0; s < 2 * M; s += 8) {
        launches += one_pass_any(skr_words / 2, src, dst, n, DigitSel{0, 32 + s, 0}, static_cast<uint32_t *>(scratch), prof, st, nullptr,
                                 s + 8 >= 2 * M ? side_out : nullptr);
        void *t = src;
        src = dst;
        dst = t;
        passes++;
    }
    *result_in_b = (src == b);
    *passes_out = passes;
    return launches;
}

// v3: 8-byte entries {key << 32 | slot} sorted on the low `key_bits` bits of the key (stable, so entries of one key keep
// their order: slots ascend with arrival).
// n_real_dev != nullptr: entries with the all-ones key (empty pieces) are dropped by the first pass; *n_real_dev (device memory) is
// the number of the others, which is what the later passes — launched for n, the host's bound — work on.
int radix_sort_entries(void *a, void *b, uint64_t n, int key_bits, void *scratch, bool *result_in_b, int *passes_out, const uint16_t *slot_info,
                       uint16_t *sorted_info, KernelProf *prof, cudaStream_t st, const unsigned long long *n_real_dev) {
    *result_in_b = false;
    *passes_out = 0;
    if (n == 0) return 0;
    int launches = 0, passes = 0;
    void *src = a, *dst = b;
    for (int s = 0; s < key_bits; s += 8) {
        const bool last = s + 8 >= key_bits;
        launches += one_pass_any(1, src, dst, n, DigitSel{0, 32 + s, 0}, static_cast<uint32_t *>(scratch), prof, st, nullptr, nullptr, last ? slot_info : nullptr,
                                 last ? sorted_info : nullptr, (n_real_dev && s > 0) ? n_real_dev : nullptr, n_real_dev && s == 0);
        void *t = src;
        src = dst;
        dst = t;
        passes++;
    }
    *result_in_b = (src == b);
    *passes_out = passes;
    return launches;
}

int radix_partition_skr_by_owner(const void *in, void *out, uint64_t n, int skr_words, uint32_t n_parts, void *scratch, uint64_t *d_counts,
                                 cudaStream_t st) {
    if (n == 0) {
        cudaMemsetAsync(d_counts, 0, sizeof(uint64_t) * n_parts, st);
        return 0;
    }
    const int nu64 = skr_words / 2;
    const int launches = one_pass_any(nu64, in, out, n, DigitSel{0, 32, n_parts}, static_cast<uint32_t *>(scratch), nullptr, st);
    part_counts_kernel<<<1, RS_RADIX, 0, st>>>(static_cast<uint32_t *>(scratch), ntiles_any(nu64, n), n_parts, n, d_counts);
    return launches + 1;
}

// Owner partition of super-k-mer records fused with the exchange: see the notes above xchg_counts_kernel.
int radix_exchange_skr_by_owner(const void *in, uint64_t n, int skr_words, void *scratch, const XchgPlan &xp, cudaStream_t st) {
    // n == 0 still takes part in the count exchange and the completion barrier (one empty tile)
    return one_pass_any(skr_words / 2, in, nullptr, n, DigitSel{0, 32, xp.world}, static_cast<uint32_t *>(scratch), nullptr, st, &xp);
}

// ------------------------------------------------------------------ one owner part (the table in parts, one part per call)
// Stable select of the records with owner_of_mmer(m-mer, n_parts) == part, written in input order to out[0..): one launch that
// reads every record once and writes only the selected ones, at their final place.  Tiles are handed out by a ticket, so a tile's
// predecessor is always running, and a tile's output offset comes from the decoupled look-back (lookback.cuh).  Inside a tile,
// record j = tile * SEL_TILE + i * SEL_THREADS + tid; the (round i, warp) counts are scanned in that order, which is input order.
// SKR: super-k-mer records (m-mer in word 1, windows in the low byte of word 2); else instance records (m-mer in the low half of
// the last 64-bit word, one window each).  counters[0] += records selected, counters[1] += their k-mer instances.
constexpr int SEL_THREADS = 256, SEL_ITEMS = 4, SEL_TILE = SEL_THREADS * SEL_ITEMS;
static_assert(SEL_ITEMS * RS_WARPS == 32, "one lane per (round, warp) count");

template <int NU64, bool SKR>
__global__ void __launch_bounds__(SEL_THREADS)
    select_part_kernel(const Blob<NU64> *__restrict__ in, uint64_t n, uint32_t part, uint32_t n_parts, Blob<NU64> *__restrict__ out,
                       unsigned long long *__restrict__ tile_state, uint32_t *__restrict__ ticket, unsigned long long *__restrict__ counters) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_off[SEL_ITEMS * RS_WARPS];
    __shared__ unsigned long long s_inst[RS_WARPS];
    __shared__ unsigned long long s_base;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t base = (uint64_t)tile * SEL_TILE;
    Blob<NU64> items[SEL_ITEMS];
    bool sel[SEL_ITEMS];
    unsigned long long inst = 0;
#pragma unroll
    for (int i = 0; i < SEL_ITEMS; i++) {
        const uint64_t j = base + (uint64_t)i * SEL_THREADS + tid;
        sel[i] = false;
        if (j < n) {
            items[i] = load_blob<NU64>(in + j);
            const uint32_t mmer = SKR ? (uint32_t)(items[i].w[0] >> 32) : (uint32_t)items[i].w[NU64 - 1];
            sel[i] = owner_of_mmer(mmer, n_parts) == part;
            if (sel[i]) inst += SKR ? (items[i].w[1] & 0xffull) : 1ull;
        }
    }
#pragma unroll
    for (int i = 0; i < SEL_ITEMS; i++) {
        const unsigned b = __ballot_sync(0xffffffffu, sel[i]);
        if (lane == 0) s_off[i * RS_WARPS + warp] = __popc(b);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) inst += __shfl_xor_sync(0xffffffffu, inst, d);
    if (lane == 0) s_inst[warp] = inst;
    __syncthreads();
    if (warp == 0) {
        const uint32_t c = s_off[lane];
        uint32_t incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += v;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        s_off[lane] = incl - c;
        if (lane == 0) lkb_publish_aggregate(tile_state, tile, total);
        const unsigned long long prefix = lkb_resolve_warp<1>(tile_state, tile, total, lane);
        if (lane == 0) {
            s_base = prefix;
            unsigned long long ti = 0;
            for (int w = 0; w < RS_WARPS; w++) ti += s_inst[w];
            if (total) atomicAdd(&counters[0], (unsigned long long)total);
            if (ti) atomicAdd(&counters[1], ti);
        }
    }
    __syncthreads();
    const unsigned long long b0 = s_base;
    const uint32_t lt_mask = (1u << lane) - 1;
#pragma unroll
    for (int i = 0; i < SEL_ITEMS; i++) {
        const unsigned b = __ballot_sync(0xffffffffu, sel[i]);
        if (sel[i]) store_blob<NU64>(out + b0 + s_off[i * RS_WARPS + warp] + __popc(b & lt_mask), items[i]);
    }
}

size_t select_part_state_bytes(uint64_t n) { return (n / SEL_TILE + 1) * sizeof(unsigned long long); }

int select_part(const void *in, uint64_t n, int rec_words, bool skr, uint32_t part, uint32_t n_parts, void *out, unsigned long long *tile_state,
                uint32_t *ticket, unsigned long long *counters, cudaStream_t st) {
    if (n == 0) return 0;
    const uint64_t tiles = (n + SEL_TILE - 1) / SEL_TILE;
    cudaMemsetAsync(tile_state, 0, tiles * sizeof(unsigned long long), st);
    cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st);
    const unsigned grid = (unsigned)tiles;
#define GBIN_SELECT(NU64, SKR)                                                                                                            \
    select_part_kernel<NU64, SKR><<<grid, SEL_THREADS, 0, st>>>(static_cast<const Blob<NU64> *>(in), n, part, n_parts, static_cast<Blob<NU64> *>(out), \
                                                                 tile_state, ticket, counters)
    if (skr) {
        if (rec_words == 8) GBIN_SELECT(4, true);
        else GBIN_SELECT(6, true);
    } else {
        if (rec_words == 4) GBIN_SELECT(2, false);
        else GBIN_SELECT(3, false);
    }
#undef GBIN_SELECT
    return 1;
}

}  // namespace gbin
