// skr_scan.cu — pipeline v2 scan stage: process_read's window/signature work (binning.c:918-1040)
// emitting one super-k-mer record per signature segment instead of one record per window.
//
// One warp per read (pack in shared memory, then the signature chain by hops i -> sig+1; a hop is a
// single REDUX.MAX over keys that carry score, inverted offset and strand bit).  Every warp works on
// tiles of RPW consecutive reads on its own (no CTA-wide barrier anywhere): it stages the records of
// the tile in shared memory, obtains the tile's global output offset from a single-pass chained scan
// over tiles (lookback.cuh; tiles are handed out in order by an atomic ticket so a predecessor is
// always running; the next ticket is already in flight while the look-back runs), and the staged
// records leave the SM as one contiguous run of 16-byte stores.
// The output is therefore in arrival order (read-major, segment-minor) and deterministic — the
// later stable sort by m-mer keeps arrival order per bucket.
#include <type_traits>

#include "gbin_device.cuh"
#include "gbin_internal.h"
#include "lookback.cuh"
#include "read_pack.cuh"
#include "skr.cuh"

namespace gbin {

constexpr int SKR_WARPS = 8;
// per warp: packed words, m-mer scores (with strand bit), segment list of the current read (2 words per segment), staged
// records; every region is a multiple of 16 bytes
__host__ __device__ inline uint32_t skr_len4(uint32_t max_len) { return (max_len + 3u) & ~3u; }
__host__ __device__ inline uint32_t skr_warp_smem(uint32_t max_len, uint32_t seg_cap, int words) {
    return 4 * scan_pk_words(max_len) + 4 * skr_len4(max_len) + 8 * skr_len4(max_len) + 4 * seg_cap * words;
}

// Per-warp scratch carved out of dynamic shared memory.
struct WarpScratch {
    uint32_t *pk, *wr, *segl, *stage;
};

// One warp tile = rpw consecutive reads handled by one warp.  DIRECT = false: records are staged in shared memory (at
// most seg_cap of them; the rest is only counted).  DIRECT = true: records are written straight to out + base (used to
// redo a tile whose segments did not fit the staging area).  Returns the number of records of the tile.
template <int PW, bool DIRECT, bool PACKED>
__device__ __forceinline__ uint32_t skr_process_tile(const ReadsView &rv, const WarpScratch &ws, uint64_t first, uint32_t rpw, int K, int M,
                                                     uint32_t arrival_base, uint32_t seg_cap, uint32_t lane, uint32_t *__restrict__ out,
                                                     unsigned long long base, uint32_t &nbad, unsigned long long &ninst) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    const uint32_t FULL = (1u << (2 * M)) - 1;
    const uint32_t C = K - M + 1;
    uint32_t nseg = 0;
    for (uint32_t rr = 0; rr < rpw; rr++) {
        const uint64_t r = first + rr;
        if (r >= rv.n_reads) break;
        const uint32_t L = rv.len(r);
        if (L < (uint32_t)K) continue;
        const uint32_t W = L - K + 1;
        const uint32_t bad = warp_pack_read(ws.pk, rv.data + rv.start(r), L, lane);
        if (!DIRECT) {
            nbad += bad;
            ninst += (lane == 0) ? W : 0;
        }
        warp_mmer_scores_strand(ws.pk, ws.wr, L, M, FULL, lane);
        const uint32_t arrival = arrival_base + (uint32_t)r;
        // phase 1: the signature chain, one hop per segment; lane 0 notes the segments of this read
        uint32_t i = 0, nsr = 0;
        while (i < W) {
            uint32_t w_rev;  // w(sig) << 1 | is_rev of the signature (binning.c:943,948)
            const uint32_t sig = i + warp_signature_hop_strand<PACKED>(ws.wr, i, C, lane, &w_rev);
            const uint32_t next = min(sig + 1, W);
            if (lane == 0) {
                ws.segl[2 * nsr] = i | ((next - i) << 16) | ((w_rev & 1u) << 24) | ((sig - i) << 25);  // sig - i <= K-M <= 62
                ws.segl[2 * nsr + 1] = w_rev >> 1;
            }
            nsr++;
            i = next;
        }
        __syncwarp();
        // phase 2: all lanes build record words, one (segment, word) pair per lane and step — no divergence
        for (uint32_t e = lane; e < nsr * NW; e += 32) {
            const uint32_t sg = e / NW, j = e - sg * NW;
            const uint32_t info = ws.segl[2 * sg], mx = ws.segl[2 * sg + 1];
            const uint32_t st0 = info & 0xffffu, n = (info >> 16) & 0xffu, rev = (info >> 24) & 1u, so = (info >> 25) & 0x3fu;
            const uint32_t jp = j >= 4 ? j - 4 : 0;
            const uint32_t bit = 2 * st0, wi = (bit >> 5) + jp, sh = bit & 31;
            uint32_t word = __funnelshift_l(ws.pk[wi + 1], ws.pk[wi], sh);
            const int keep = 2 * (int)(K + n - 1) - 32 * (int)jp;  // valid payload bits in this word
            word = keep >= 32 ? word : (keep <= 0 ? 0u : (word & (0xffffffffu << (32 - keep))));
            word = j == 0 ? arrival : (j == 1 ? mx : (j == 2 ? (n | (rev << 8) | (so << 16)) : (j == 3 ? st0 : word)));
            if (DIRECT) out[(base + nseg + sg) * NW + j] = word;
            else if (nseg + sg < seg_cap) ws.stage[(nseg + sg) * NW + j] = word;
        }
        nseg += nsr;
        __syncwarp();
    }
    return nseg;
}

template <int PW, bool PACKED>
__global__ void __launch_bounds__(SKR_WARPS * 32)
    skr_scan_kernel(ReadsView rv, uint64_t read_begin, int K, int M, uint32_t arrival_base, uint32_t max_len, uint32_t rpw, uint32_t seg_cap,
                    uint32_t ntiles, uint32_t *__restrict__ out, unsigned long long capacity, unsigned long long *__restrict__ tile_state,
                    uint32_t *__restrict__ ticket, unsigned long long *__restrict__ counters /* [0] bad bases, [1] records, [2] instances */,
                    uint32_t lkb_sleep) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *wbase = smem + (size_t)warp * skr_warp_smem(max_len, seg_cap, NW);
    WarpScratch ws;
    ws.pk = reinterpret_cast<uint32_t *>(wbase);
    ws.wr = ws.pk + scan_pk_words(max_len);
    ws.segl = ws.wr + skr_len4(max_len);  // per segment of the current read: start | n << 16 | rev << 24, m-mer code
    ws.stage = ws.segl + 2 * skr_len4(max_len);
    uint32_t nbad = 0;
    unsigned long long ninst = 0;
    // records emitted by earlier launches over the same batch (the host path scans the reads in chunks while later
    // chunks are still on their way over PCIe); rv.n_reads is the END of this launch's read range
    const unsigned long long base0 = counters[1];

    uint32_t tile = 0;
    if (lane == 0) tile = atomicAdd(ticket, 1u);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    while (tile < ntiles) {
        const uint64_t first = read_begin + (uint64_t)tile * rpw;
        const uint32_t nseg = skr_process_tile<PW, false, PACKED>(rv, ws, first, rpw, K, M, arrival_base, seg_cap, lane, out, 0ull, nbad, ninst);
        if (lane == 0) lkb_publish_aggregate(tile_state, tile, nseg);
        const unsigned long long base = base0 + lkb_resolve_warp<1>(tile_state, tile, nseg, lane, lkb_sleep);
        if (tile == ntiles - 1 && lane == 0) counters[1] = base + nseg;
        if (base + nseg <= capacity) {  // past the capacity only the total is produced (the caller re-runs)
            if (nseg <= seg_cap) {
                uint4 *dst = reinterpret_cast<uint4 *>(out + base * NW);
                const uint4 *src = reinterpret_cast<const uint4 *>(ws.stage);
                const uint32_t nvec = nseg * (NW / 4);
                for (uint32_t v = lane; v < nvec; v += 32) dst[v] = src[v];
            } else {  // more segments than the staging area holds (rare): redo the tile, writing in place
                (void)skr_process_tile<PW, true, PACKED>(rv, ws, first, rpw, K, M, arrival_base, seg_cap, lane, out, base, nbad, ninst);
            }
        }
        // the next ticket is taken only now: a ticket taken before the look-back lets later tiles overtake this warp's next
        // tile, and their resolve then waits for it (measured: 1.5x slower)
        uint32_t next_tile = 0;
        if (lane == 0) next_tile = atomicAdd(ticket, 1u);
        tile = __shfl_sync(0xffffffffu, next_tile, 0);
    }
    if (nbad) atomicAdd(&counters[0], (unsigned long long)nbad);
    if (ninst) atomicAdd(&counters[2], ninst);
}

// ---------------------------------------------------------------------------------------------------------------------
// Scan kernel B (reads of at most 32 * NJ m-mer positions, NJ <= 8): one lane per m-mer position.
//
// The hop chain of the kernel above spends one REDUX round trip per segment.  Here the leftmost arg-max A(i) of the
// m-mer scores over [i, i + C) is computed for ALL windows of a read at once: every lane holds the keys
// {w(p) << 9 | (255 - p) << 1 | is_rev(p)} of positions p = lane + 32 j in registers, and a sliding maximum of width C is
// built from widths 1, 2, 4, ... by shuffles (max is idempotent, so the last step may overlap: width C = max of two
// width-2^b windows C - 2^b apart).  The inverted position below the score makes the maximum the LEFTMOST best position
// (binning.c:972 replaces the signature only on a strictly larger score).  A(i) goes to shared memory as one byte per
// window.  The chain i -> A(i) + 1 (binning.c:922: a signature is kept until the window start passes it) is then walked
// by ONE LANE PER READ for the rpw reads of the tile in parallel, first to count the tile's segments (the count feeds the
// chained scan over tiles), then to list them.  Records are built one lane per segment (header + payload words from the
// packed read) and written straight to their final place with 16-byte stores: neighbouring lanes write neighbouring
// records, so there is no staging copy.
// Value of lane + d.  Past the last lane the result is garbage (the caller's own value), which is harmless here: a window
// that starts at a real window start i < W ends at position i + C - 1 <= L - M, inside the 32 lanes, so garbage only ever
// reaches the outputs of window starts that do not exist.
template <typename KeyT>
__device__ __forceinline__ KeyT s2_down(KeyT v, uint32_t d, uint32_t) {
    return __shfl_down_sync(0xffffffffu, v, d);
}
template <typename KeyT>
__device__ __forceinline__ KeyT s2_max(KeyT a, KeyT b) { return a > b ? a : b; }

// Sliding maximum of width C over the keys of a read, lane l holding positions PL*l .. PL*l + PL-1 in x[] (C >= PL).
// In: x[a] = key of position PL*l + a.  Out: x[a] = max over [PL*l + a, PL*l + a + C).  With C - PL = F0*PL + B0 the window
// of position PL*l + a is: the lane's own suffix from a, then F whole lanes, then the first b positions of lane l + F + 1,
// where (F, b) = (F0, B0 + a) if B0 + a < PL, else (F0 + 1, B0 + a - PL).  Whole-lane ranges come from a doubling over the
// per-lane maxima (one register per step instead of PL), prefixes and suffixes are local.  B0 is a template parameter so that
// every register index is static.
template <int PL, int B0, typename KeyT>
__device__ __forceinline__ void s2_window_max(KeyT (&x)[PL], uint32_t F0, uint32_t lane) {
    KeyT pre[PL], suf[PL];
    pre[0] = x[0];
#pragma unroll
    for (int a = 1; a < PL; a++) pre[a] = s2_max(pre[a - 1], x[a]);
    suf[PL - 1] = x[PL - 1];
#pragma unroll
    for (int a = PL - 2; a >= 0; a--) suf[a] = s2_max(suf[a + 1], x[a]);
    const KeyT m = pre[PL - 1];
    KeyT mm = m;  // max over lanes [l, l + w)
    uint32_t w = 1;
    for (; 2 * w <= F0; w *= 2) mm = s2_max(mm, s2_down(mm, w, lane));
    KeyT full0 = 0;  // lanes l+1 .. l+F0
    if (F0) {
        full0 = s2_down(mm, 1, lane);
        if (F0 > w) full0 = s2_max(full0, s2_down(mm, 1 + F0 - w, lane));
    }
    KeyT full1 = full0;  // lanes l+1 .. l+F0+1
    if (B0 > 0) full1 = s2_max(full0, s2_down(m, F0 + 1, lane));
#pragma unroll
    for (int a = 0; a < PL; a++) {
        const int t = B0 + a;
        KeyT r;
        if (t < PL) {
            r = s2_max(suf[a], full0);
            if (t > 0) r = s2_max(r, s2_down(pre[t > 0 ? t - 1 : 0], F0 + 1, lane));
        } else {
            r = s2_max(suf[a], full1);
            if (t - PL > 0) r = s2_max(r, s2_down(pre[t - PL > 0 ? t - PL - 1 : 0], F0 + 2, lane));
        }
        x[a] = r;
    }
}
template <int PL, typename KeyT, int B = 0>
__device__ __forceinline__ void s2_window_max_sel(KeyT (&x)[PL], uint32_t b0, uint32_t F0, uint32_t lane) {
    if constexpr (B < PL) {
        if (b0 == (uint32_t)B) s2_window_max<PL, B, KeyT>(x, F0, lane);
        else s2_window_max_sel<PL, KeyT, B + 1>(x, b0, F0, lane);
    }
}

__host__ __device__ inline uint32_t s2_pk_words(uint32_t max_len) { return scan_pk_words(max_len) | 1u; }  // odd: reads fall into different banks
__host__ __device__ inline uint32_t s2_sig_bytes(int nj) { return 32u * (uint32_t)nj + 4u; }                 // odd number of words
__host__ __device__ inline uint32_t s2_warp_smem(uint32_t max_len, int nj, uint32_t rpw, uint32_t seg_cap) {
    return (4u * s2_pk_words(max_len) * rpw + s2_sig_bytes(nj) * rpw + 4u * seg_cap + 15u) & ~15u;
}

#ifndef S2_LKB_DEPTH
#define S2_LKB_DEPTH 4
#endif
template <int PW, int NJ, typename KeyT>
__global__ void __launch_bounds__(SKR_WARPS * 32)
    skr_scan2_kernel(ReadsView rv, uint64_t read_begin, int K, int M, uint32_t arrival_base, uint32_t max_len, uint32_t rpw, uint32_t seg_cap,
                     uint32_t ntiles, uint32_t *__restrict__ out, unsigned long long capacity, unsigned long long *__restrict__ tile_state,
                     uint32_t *__restrict__ ticket, unsigned long long *__restrict__ counters /* [0] bad bases, [1] records, [2] instances */,
                     uint32_t lkb_sleep) {
    constexpr int NW = SkrLayout<PW>::WORDS;
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t pkw = s2_pk_words(max_len), sgb = s2_sig_bytes(NJ);
    uint8_t *wbase = smem + (size_t)warp * s2_warp_smem(max_len, NJ, rpw, seg_cap);
    uint32_t *pk = reinterpret_cast<uint32_t *>(wbase);
    uint32_t *segl = pk + pkw * rpw;
    uint8_t *sig = reinterpret_cast<uint8_t *>(segl + seg_cap);
    const uint32_t FULL = (1u << (2 * M)) - 1;
    const uint32_t C = K - M + 1;
    const uint32_t down = 32u - 2u * (uint32_t)M;
    const uint32_t win_f0 = (C - NJ) / NJ, win_b0 = (C - NJ) % NJ;  // C >= NJ (the launcher sees to it)
    uint32_t nbad = 0;
    unsigned long long ninst = 0;
    const unsigned long long base0 = counters[1];  // records of earlier launches over the same batch (chunked host feed)

    uint32_t tile = 0;
    if (lane == 0) tile = atomicAdd(ticket, 1u);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    while (tile < ntiles) {
        const uint64_t first = read_begin + (uint64_t)tile * rpw;
        // ---- phase A, the warp over one read at a time: pack, score, sliding arg-max
        // lane q holds start and length of read first + q (length 0: past the end of the range, or shorter than K)
        uint64_t my_start = 0;
        uint32_t myL = 0;
        if (lane < rpw && first + lane < rv.n_reads) {
            myL = rv.len(first + lane);
            my_start = rv.start(first + lane);
            if (myL < (uint32_t)K) myL = 0;
        }
        const uint32_t myW = myL ? myL - K + 1 : 0;
        // the loads of read rr + 1 are issued before read rr is worked on
        uint32_t nw0 = 0, nw31 = 0;
        uint32_t nL = __shfl_sync(0xffffffffu, myL, 0);
        uint64_t nstart = __shfl_sync(0xffffffffu, my_start, 0);
        if (nL) warp_pack_load(rv.data + nstart, nL, 0, lane, nw0, nw31);
        for (uint32_t rr = 0; rr < rpw; rr++) {
            const uint32_t L = nL, w0 = nw0, w31 = nw31;
            const uint8_t *src = rv.data + nstart;
            if (rr + 1 < rpw) {
                nL = __shfl_sync(0xffffffffu, myL, rr + 1);
                nstart = __shfl_sync(0xffffffffu, my_start, rr + 1);
                if (nL) warp_pack_load(rv.data + nstart, nL, 0, lane, nw0, nw31);
            }
            if (!L) continue;
            uint32_t *pkr = pk + rr * pkw;
            {
                const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3u);
                nbad += warp_pack_chunk(pkr, w0, w31, mis, L, 0, lane);
                uint32_t nchunks = 1;
                for (uint32_t c0 = 128; c0 < L; c0 += 128, nchunks++) {
                    uint32_t v0, v31;
                    warp_pack_load(src, L, c0, lane, v0, v31);
                    nbad += warp_pack_chunk(pkr, v0, v31, mis, L, c0, lane);
                }
                if (lane < PK_PAD_WORDS) pkr[8 * nchunks + lane] = 0u;
                __syncwarp();
            }
            KeyT x[NJ];  // keys of positions NJ * lane + a
            {
                // the 64 packed bits from position p0 on, then one static funnel shift per position.  Positions past L - M get
                // keys made of the zero padding: they only reach windows that do not exist (see s2_down).
                const uint32_t p0 = NJ * lane, bit0 = 2 * p0, wi = bit0 >> 5, sh0 = bit0 & 31;
                const uint32_t q0 = pkr[wi], q1 = pkr[wi + 1], q2 = pkr[wi + 2];
                const uint32_t v0 = __funnelshift_l(q1, q0, sh0), v1 = __funnelshift_l(q2, q1, sh0);
                const uint32_t lob = ((255u - p0) << 1) | 1u;
#pragma unroll
                for (int a = 0; a < NJ; a++) {
                    const uint32_t s = __funnelshift_l(v1, v0, 2 * a) >> down;
                    // c = FULL - s = FULL ^ s scores higher iff the top bit of s is clear (binning.c:943,948: strictly higher)
                    const uint32_t top = s >> (2 * M - 1);              // 1: forward strand kept
                    const uint32_t mx = s ^ ((top - 1u) & FULL);        // max(s, FULL - s)
                    x[a] = ((KeyT)mx << 9) | ((lob - 2u * a) ^ top);   // ... | (255 - p) << 1 | is_rev
                }
            }
            s2_window_max_sel<NJ, KeyT>(x, win_b0, win_f0, lane);
            uint8_t *sg = sig + rr * sgb + NJ * lane;  // stored inverted: 255 - A(i)
#pragma unroll
            for (int a = 0; a < NJ; a++) sg[a] = (uint8_t)((uint32_t)x[a] >> 1);
        }
        __syncwarp();
        ninst += myW;
        // ---- phase B, one lane per read: count the segments of the chain i -> A(i) + 1
        const uint8_t *sg = sig + lane * sgb;
        uint32_t cnt = 0;
        for (uint32_t i = 0; i < myW; cnt++) i = min(256u - (uint32_t)sg[i], myW);
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += up;
        }
        const uint32_t off = incl - cnt, nseg = __shfl_sync(0xffffffffu, incl, 31);
        if (lane == 0) lkb_publish_aggregate(tile_state, tile, nseg);
        // a window of 128 predecessors per step: a step is one round trip to L2, and with thousands of warps finishing tiles
        // every few ns a 32-wide walk falls behind the tiles that publish meanwhile (measured: ~40 steps per tile)
        const unsigned long long base = base0 + lkb_resolve_warp<S2_LKB_DEPTH>(tile_state, tile, nseg, lane, lkb_sleep);
        if (tile == ntiles - 1 && lane == 0) counters[1] = base + nseg;
        if (base + nseg <= capacity) {  // past the capacity only the total is produced (the caller re-runs)
            // ---- phase C: list the segments (seg_cap at a time), then one lane per segment builds and stores its record
            for (uint32_t lo = 0; lo < nseg; lo += seg_cap) {
                uint32_t g = off;
                for (uint32_t i = 0; i < myW; g++) {
                    const uint32_t sp = 255u - (uint32_t)sg[i], nx = min(sp + 1u, myW);
                    if (g - lo < seg_cap) segl[g - lo] = lane | (i << 8) | (sp << 16) | ((nx - i) << 24);  // g < lo wraps around: not stored
                    i = nx;
                }
                __syncwarp();
                const uint32_t cw = min(seg_cap, nseg - lo);
                for (uint32_t e = lane; e < cw; e += 32) {
                    const uint32_t info = segl[e];
                    const uint32_t rr = info & 0xffu, st0 = (info >> 8) & 0xffu, sp = (info >> 16) & 0xffu, n = info >> 24;
                    const uint32_t *pkr = pk + rr * pkw;
                    uint32_t bit = 2 * sp, wi = bit >> 5, sh = bit & 31;
                    const uint32_t s = __funnelshift_l(pkr[wi + 1], pkr[wi], sh) >> down;
                    const uint32_t c = FULL - s;
                    uint32_t w[NW];
                    w[0] = arrival_base + (uint32_t)(first + rr);
                    w[1] = c > s ? c : s;
                    w[2] = n | ((c > s ? 1u : 0u) << 8) | ((sp - st0) << 16);
                    w[3] = st0;
                    bit = 2 * st0, wi = bit >> 5, sh = bit & 31;
                    uint32_t prev = pkr[wi];
#pragma unroll
                    for (int jp = 0; jp < NW - 4; jp++) {
                        const uint32_t nxw = pkr[wi + jp + 1];
                        const uint32_t word = __funnelshift_l(nxw, prev, sh);
                        prev = nxw;
                        const int keep = 2 * (int)(K + n - 1) - 32 * jp;  // valid payload bits in this word
                        w[4 + jp] = keep >= 32 ? word : (keep <= 0 ? 0u : (word & (0xffffffffu << (32 - keep))));
                    }
                    uint4 *dst = reinterpret_cast<uint4 *>(out + (base + lo + e) * NW);
#pragma unroll
                    for (int v = 0; v < NW / 4; v++) dst[v] = make_uint4(w[4 * v], w[4 * v + 1], w[4 * v + 2], w[4 * v + 3]);
                }
                __syncwarp();
            }
        }
        uint32_t next_tile = 0;
        if (lane == 0) next_tile = atomicAdd(ticket, 1u);
        tile = __shfl_sync(0xffffffffu, next_tile, 0);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        nbad += __shfl_xor_sync(0xffffffffu, nbad, d);
        ninst += __shfl_xor_sync(0xffffffffu, ninst, d);
    }
    if (lane == 0 && nbad) atomicAdd(&counters[0], (unsigned long long)nbad);
    if (lane == 0 && ninst) atomicAdd(&counters[2], ninst);
}

// Shape of kernel B for a batch, or nj = 0 when the reads are too long for it (more than 256 m-mer positions).
struct Scan2Shape {
    int nj;
    bool wide;  // 64-bit keys: score, position and strand bit do not fit 32 bits (M > 11)
    uint32_t rpw, seg_cap;
};
static Scan2Shape skr_scan2_shape(int K, int M, uint32_t max_len) {
    Scan2Shape sh{0, false, 0, 0};
    if (max_len < (uint32_t)K) return sh;
    const uint32_t npos = max_len - M + 1;
    if (npos > 256u) return sh;
    sh.nj = npos <= 96u ? 3 : (npos <= 160u ? 5 : 8);
    if (K - M + 1 < sh.nj) return Scan2Shape{0, false, 0, 0};  // the window must span at least one lane's positions
    sh.wide = 2 * M + 9 > 32;
    const uint32_t W = max_len - K + 1;
    uint32_t per_read = (uint32_t)(1.6 * (double)W / ((K - M + 2) / 2.0)) + 2;
    if (per_read > W) per_read = W;
    const uint32_t bytes_per_read = 4u * s2_pk_words(max_len) + s2_sig_bytes(sh.nj) + 4u * per_read;
    uint32_t rpw = 8192u / bytes_per_read;
    if (rpw > 32u) rpw = 32u;
    if (rpw < 4u) rpw = 4u;
    sh.rpw = rpw;
    sh.seg_cap = (rpw * per_read + 3u) & ~3u;
    return sh;
}

// Tile shape: rpw reads per warp and a staging area of seg_cap records, sized for 1.6x the expected number of segments
// (a segment covers about (K-M+2)/2 windows) within a budget of SKR_STAGE_BYTES per warp; tiles that exceed it are redone in place.
constexpr uint32_t SKR_STAGE_BYTES = 6144;
static void skr_tile_shape(int K, int M, uint32_t max_len, uint32_t *rpw_out, uint32_t *seg_cap_out) {
    const int NW = skr_words(K);
    const uint32_t W = max_len >= (uint32_t)K ? max_len - K + 1 : 1;
    const uint32_t budget = SKR_STAGE_BYTES / (NW * 4u);  // records
    uint32_t per_read = (uint32_t)(1.6 * (double)W / ((K - M + 2) / 2.0)) + 2;
    if (per_read > W) per_read = W;
    uint32_t rpw = budget / per_read;
    if (rpw < 1) rpw = 1;
    if (rpw > SKR_STAGE_BYTES / 512u) rpw = SKR_STAGE_BYTES / 512u;  // 12 reads per tile
    uint32_t cap = rpw * per_read;
    if (cap > budget) cap = budget;
    if (cap < 4) cap = 4;
    *rpw_out = rpw;
    *seg_cap_out = cap;
}

// ns between polls of a predecessor tile that has not published yet: the kernel is bound by instruction issue, so a
// spinning warp takes issue slots from the warps that still compute
constexpr uint32_t SKR_POLL_SLEEP_NS = 800;

// Host launcher.  tile_state must hold skr_scan_tiles() u64 (zeroed here), ticket one u32 (zeroed here).
// Returns kernels launched.
int launch_skr_scan(const ReadsView &rv_all, uint64_t read_begin, uint64_t read_end, int K, int M, uint32_t arrival_base, uint32_t max_len,
                    void *out, uint64_t capacity, unsigned long long *tile_state, uint32_t *ticket, unsigned long long *counters, int sm_count,
                    cudaStream_t st) {
    if (read_end <= read_begin) return 0;
    ReadsView rv = rv_all;
    rv.n_reads = read_end;  // the kernel treats n_reads as the end of its read range
    const int PW = skr_payload_units(K);
    const int NW = 4 + 2 * PW;
    const Scan2Shape s2 = skr_scan2_shape(K, M, max_len);
    if (s2.nj) {
        const uint32_t ntiles = (uint32_t)((read_end - read_begin + s2.rpw - 1) / s2.rpw);
        const size_t smem = (size_t)SKR_WARPS * s2_warp_smem(max_len, s2.nj, s2.rpw, s2.seg_cap);
        cudaMemsetAsync(tile_state, 0, sizeof(unsigned long long) * ntiles, st);
        cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st);
        uint32_t blocks = (uint32_t)sm_count * 8;
        if (blocks > (ntiles + SKR_WARPS - 1) / SKR_WARPS) blocks = (ntiles + SKR_WARPS - 1) / SKR_WARPS;
        bool failed = false;
        auto launch = [&](auto kern) {
            if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
                (void)cudaGetLastError();
                failed = true;
                return;
            }
            kern<<<blocks, SKR_WARPS * 32, smem, st>>>(rv, read_begin, K, M, arrival_base, max_len, s2.rpw, s2.seg_cap, ntiles, static_cast<uint32_t *>(out),
                                                       capacity, tile_state, ticket, counters, SKR_POLL_SLEEP_NS);
        };
        auto pick_nj = [&](auto pw, auto key) {
            constexpr int P = decltype(pw)::value;
            using KeyT = decltype(key);
            if (s2.nj == 3) launch(skr_scan2_kernel<P, 3, KeyT>);
            else if (s2.nj == 5) launch(skr_scan2_kernel<P, 5, KeyT>);
            else launch(skr_scan2_kernel<P, 8, KeyT>);
        };
        if (PW == 2) {
            if (s2.wide) pick_nj(std::integral_constant<int, 2>{}, (unsigned long long)0);
            else pick_nj(std::integral_constant<int, 2>{}, (uint32_t)0);
        } else {
            if (s2.wide) pick_nj(std::integral_constant<int, 4>{}, (unsigned long long)0);
            else pick_nj(std::integral_constant<int, 4>{}, (uint32_t)0);
        }
        if (!failed) return 1;
    }
    uint32_t rpw, seg_cap;
    skr_tile_shape(K, M, max_len, &rpw, &seg_cap);
    const uint32_t ntiles = (uint32_t)((read_end - read_begin + rpw - 1) / rpw);
    // long reads need more shared memory per warp: fewer warps per block then (-1: not even one fits; the caller uses the other scan kernel)
    int dev = 0, limit = 48 * 1024;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const size_t per_warp = skr_warp_smem(max_len, seg_cap, NW);
    int warps = SKR_WARPS;
    while (warps > 1 && (size_t)warps * per_warp > (size_t)limit) warps >>= 1;
    if ((size_t)warps * per_warp > (size_t)limit) return -1;
    const size_t smem = (size_t)warps * per_warp;
    cudaMemsetAsync(tile_state, 0, sizeof(unsigned long long) * ntiles, st);
    cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st);
    uint32_t blocks = (uint32_t)sm_count * 8;
    if (blocks > (ntiles + warps - 1) / warps) blocks = (ntiles + warps - 1) / warps;
    // one-REDUX hops need score, inverted offset and strand bit in 32 bits (read_pack.cuh)
    const bool packed = 2 * M + 1 + ((K - M + 1) <= 32 ? 5 : 6) <= 32;
    bool attr_failed = false;
    auto launch = [&](auto kern) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            (void)cudaGetLastError();
            attr_failed = true;
            return;
        }
        kern<<<blocks, warps * 32, smem, st>>>(rv, read_begin, K, M, arrival_base, max_len, rpw, seg_cap, ntiles, static_cast<uint32_t *>(out),
                                                   capacity, tile_state, ticket, counters, SKR_POLL_SLEEP_NS);
    };
    if (PW == 2) {
        if (packed) launch(skr_scan_kernel<2, true>);
        else launch(skr_scan_kernel<2, false>);
    } else {
        if (packed) launch(skr_scan_kernel<4, true>);
        else launch(skr_scan_kernel<4, false>);
    }
    return attr_failed ? -1 : 1;
}

uint32_t skr_scan_tiles(uint64_t n_reads, int K, int M, uint32_t max_len) {
    uint32_t rpw, seg_cap;
    skr_tile_shape(K, M, max_len, &rpw, &seg_cap);
    const Scan2Shape s2 = skr_scan2_shape(K, M, max_len);
    if (s2.nj && s2.rpw < rpw) rpw = s2.rpw;  // enough for either kernel
    return (uint32_t)((n_reads + rpw - 1) / rpw);
}

}  // namespace gbin
