// gbin_device.cuh — shared device-side types for the binning kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace gbin {

// One k-mer instance = one window of one read, as process_read inserts it (binning.c:1023-1069):
// oriented k-mer code, m-mer bucket code, arrival index of the read.
// KW = 64-bit words per k-mer code (1: K <= 32, 2: K <= 64); most significant word first.
template <int KW>
struct Rec;

template <>
struct __align__(16) Rec<1> {
    uint64_t k[1];
    uint32_t mmer;
    uint32_t arrival;
};

template <>
struct __align__(8) Rec<2> {
    uint64_t k[2];
    uint32_t mmer;
    uint32_t arrival;
};

static_assert(sizeof(Rec<1>) == 16, "record layout");
static_assert(sizeof(Rec<2>) == 24, "record layout");

template <int KW>
__device__ __forceinline__ bool same_key(const Rec<KW> &a, const Rec<KW> &b) {
    bool eq = a.mmer == b.mmer;
#pragma unroll
    for (int w = 0; w < KW; w++) eq = eq && (a.k[w] == b.k[w]);
    return eq;
}

template <int KW>
__device__ __forceinline__ Rec<KW> load_rec(const Rec<KW> *p) {
    return *p;
}
template <>
__device__ __forceinline__ Rec<1> load_rec<1>(const Rec<1> *p) {
    const uint4 v = *reinterpret_cast<const uint4 *>(p);
    Rec<1> r;
    r.k[0] = (uint64_t)v.x | ((uint64_t)v.y << 32);
    r.mmer = v.z;
    r.arrival = v.w;
    return r;
}
template <int KW>
__device__ __forceinline__ void store_rec(Rec<KW> *p, const Rec<KW> &r) {
    *p = r;
}
template <>
__device__ __forceinline__ void store_rec<1>(Rec<1> *p, const Rec<1> &r) {
    *reinterpret_cast<uint4 *>(p) = make_uint4((uint32_t)r.k[0], (uint32_t)(r.k[0] >> 32), r.mmer, r.arrival);
}

// How the reads are laid out (mirror of gbin_reads in include/gbin.h, device pointers).
struct ReadsView {
    const uint8_t *data;
    uint64_t data_bytes;
    uint64_t n_reads;
    uint64_t stride;
    uint32_t read_len;
    const uint64_t *starts;  // nullptr: fixed stride
    const uint32_t *lens;
    __device__ __forceinline__ uint64_t start(uint64_t r) const { return starts ? starts[r] : r * stride; }
    __device__ __forceinline__ uint32_t len(uint64_t r) const { return lens ? lens[r] : read_len; }
};

// Owner of an m-mer bucket among `parts` GPUs: a multiplicative hash of the code, range-reduced by a multiply-shift.  Not
// `code % parts`: signatures are max-score m-mers, their last bases are far from uniform, and the plain remainder left the
// busiest of 8 owners with 4.9 % more k-mer instances than the mean (1.4 % with the hash).
__host__ __device__ inline uint32_t owner_of_mmer(uint32_t mmer_code, uint32_t parts) {
    return (uint32_t)(((uint64_t)(mmer_code * 0x9E3779B1u) * parts) >> 32);
}

}  // namespace gbin
