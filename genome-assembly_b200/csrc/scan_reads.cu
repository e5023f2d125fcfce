// scan_reads.cu — process_read's per-read work (binning.c:918-1040) as one warp per read:
//   1. ASCII -> 2-bit codes (getval map A=3 C=2 G=1 T=0, binning.c:91-111), packed MSB-first in smem;
//   2. the signature chain: at a restart window i the signature is the LEFTMOST m-mer position
//      p in [i, i+K-M] maximising w(p) = max(s(p), 4^M-1-s(p)) (binning.c:931-988, strict '>' at :972),
//      and it is kept for every following window until the window start passes it (binning.c:922;
//      the else-branch loop at :997 never runs for K >= 2M).  So the chain hops i -> sig+1: one
//      warp-wide arg-max (REDUX max + REDUX min) per hop instead of the reference's per-window scan;
//   3. per window: oriented k-mer code (bitwise complement when the signature's complement won,
//      binning.c:1029-1040 — the reference complements without reversing), m-mer code = w(sig).
// Output: one Rec<KW> per window, in arrival order (read-major, window-minor).
#include "gbin_device.cuh"
#include "gbin_internal.h"
#include "read_pack.cuh"

namespace gbin {

constexpr int SCAN_WARPS = 8;

// per warp: packed words, m-mer scores w(p), per-window info
__host__ __device__ inline uint32_t scan_warp_smem(uint32_t max_len) { return 4 * scan_pk_words(max_len) + 4 * max_len + 4 * max_len + 16; }

// windows per read (ragged form) -> u32, consumed by exclusive_scan
__global__ void count_windows_kernel(ReadsView rv, int K, uint32_t *__restrict__ counts) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rv.n_reads) return;
    const uint32_t L = rv.len(r);
    counts[r] = L >= (uint32_t)K ? L - K + 1 : 0;
}

template <int KW>
__device__ __forceinline__ void kmer_at(const uint32_t *pk, uint32_t q, int K, bool rev, uint64_t (&out)[KW]) {
    const uint32_t bit = 2 * q, wi = bit >> 5, sh = bit & 31;
    if (KW == 1) {
        const uint32_t a = __funnelshift_l(pk[wi + 1], pk[wi], sh);
        const uint32_t b = __funnelshift_l(pk[wi + 2], pk[wi + 1], sh);
        uint64_t x = (((uint64_t)a << 32) | b) >> (64 - 2 * K);
        if (rev) x = ~x & (K == 32 ? ~0ull : ((1ull << (2 * K)) - 1));
        out[0] = x;
    } else {
        const uint32_t a = __funnelshift_l(pk[wi + 1], pk[wi], sh);
        const uint32_t b = __funnelshift_l(pk[wi + 2], pk[wi + 1], sh);
        const uint32_t c = __funnelshift_l(pk[wi + 3], pk[wi + 2], sh);
        const uint32_t d = __funnelshift_l(pk[wi + 4], pk[wi + 3], sh);
        uint64_t hi = ((uint64_t)a << 32) | b, lo = ((uint64_t)c << 32) | d;
        const int r = 128 - 2 * K;  // 0..62 for 33 <= K <= 64
        if (r) {
            lo = (lo >> r) | (hi << (64 - r));
            hi >>= r;
        }
        if (rev) {
            hi = ~hi & (K == 64 ? ~0ull : ((1ull << (2 * K - 64)) - 1));
            lo = ~lo;
        }
        out[0] = hi;
        out[KW - 1] = lo;
    }
}

template <int KW>
__global__ void __launch_bounds__(SCAN_WARPS * 32)
    scan_reads_kernel(ReadsView rv, const uint64_t *__restrict__ rec_off, int K, int M, uint32_t arrival_base, uint32_t max_len,
                      Rec<KW> *__restrict__ out, unsigned long long *__restrict__ bad_bases) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *wbase = smem + (size_t)warp * scan_warp_smem(max_len);
    uint32_t *pk = reinterpret_cast<uint32_t *>(wbase);
    uint32_t *wv = pk + scan_pk_words(max_len);
    uint32_t *winfo = wv + max_len;
    const uint32_t FULL = (1u << (2 * M)) - 1;
    const uint32_t C = K - M + 1;  // m-mer positions per window
    const uint32_t wpb = blockDim.x >> 5;  // warps per block: fewer than SCAN_WARPS when long reads need more shared memory per warp
    const uint64_t warps_total = (uint64_t)gridDim.x * wpb;
    uint32_t nbad = 0;

    for (uint64_t r = (uint64_t)blockIdx.x * wpb + warp; r < rv.n_reads; r += warps_total) {
        const uint32_t L = rv.len(r);
        if (L < (uint32_t)K) continue;
        const uint32_t W = L - K + 1;
        const uint8_t *src = rv.data + rv.start(r);
        // ---- pack 16 bases per word (aligned 32-bit loads, byte-parallel conversion), then all m-mer scores
        nbad += warp_pack_read(pk, src, L, lane);
        warp_mmer_scores(pk, wv, L, M, FULL, lane);
        // ---- signature chain: hop from restart window to restart window
        uint32_t i = 0;
        while (i < W) {
            uint32_t mx;
            const uint32_t sig = warp_signature_hop(wv, i, C, lane, &mx);
            const uint32_t s_sig = mmer_at(pk, sig, M);
            const uint32_t info = (mx << 1) | (s_sig != mx ? 1u : 0u);  // bit0 = is_rev (binning.c:943,948)
            const uint32_t next = min(sig + 1, W);
            for (uint32_t q = i + lane; q < next; q += 32) winfo[q] = info;
            i = next;
        }
        __syncwarp();
        // ---- one record per window
        const uint64_t o = rec_off ? rec_off[r] : r * (uint64_t)W;
        const uint32_t arrival = arrival_base + (uint32_t)r;
        for (uint32_t q = lane; q < W; q += 32) {
            const uint32_t info = winfo[q];
            Rec<KW> rec;
            kmer_at<KW>(pk, q, K, info & 1u, rec.k);
            rec.mmer = info >> 1;
            rec.arrival = arrival;
            store_rec<KW>(out + o + q, rec);
        }
        __syncwarp();
    }
    if (nbad) atomicAdd(bad_bases, (unsigned long long)nbad);
}

// ------------------------------------------------------------------ host launchers

int launch_count_windows(const ReadsView &rv, int K, uint32_t *counts, cudaStream_t st) {
    if (rv.n_reads == 0) return 0;
    const unsigned blocks = (unsigned)((rv.n_reads + 255) / 256);
    count_windows_kernel<<<blocks, 256, 0, st>>>(rv, K, counts);
    return 1;
}

// Returns the kernels launched, or -1 when a read is too long for the shared memory of even one warp per block
// (the caller reports GBIN_E_TOO_LARGE with gbin_max_read_len()).
int launch_scan_reads(const ReadsView &rv, const uint64_t *rec_off, int K, int M, int KW, uint32_t arrival_base, uint32_t max_len,
                      void *out, unsigned long long *bad_bases, int sm_count, cudaStream_t st) {
    if (rv.n_reads == 0) return 0;
    int dev = 0, limit = 48 * 1024;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const size_t per_warp = scan_warp_smem(max_len);
    int warps = SCAN_WARPS;
    while (warps > 1 && (size_t)warps * per_warp > (size_t)limit) warps >>= 1;
    if ((size_t)warps * per_warp > (size_t)limit) return -1;
    const size_t smem = (size_t)warps * per_warp;
    uint64_t blocks = (rv.n_reads + warps - 1) / warps;
    const uint64_t cap = (uint64_t)sm_count * 8;
    if (blocks > cap) blocks = cap;
    cudaError_t e = cudaSuccess;
    if (KW == 1) {
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(scan_reads_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return -1;
        scan_reads_kernel<1><<<(unsigned)blocks, warps * 32, smem, st>>>(rv, rec_off, K, M, arrival_base, max_len, static_cast<Rec<1> *>(out), bad_bases);
    } else {
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(scan_reads_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return -1;
        scan_reads_kernel<2><<<(unsigned)blocks, warps * 32, smem, st>>>(rv, rec_off, K, M, arrival_base, max_len, static_cast<Rec<2> *>(out), bad_bases);
    }
    return 1;
}

// Longest read the v1 scan kernel holds with one warp per block.
uint32_t scan_reads_max_len() {
    int dev = 0, limit = 48 * 1024;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    uint32_t lo = 1, hi = 1u << 20;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (scan_warp_smem(mid) <= (size_t)limit) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

}  // namespace gbin
