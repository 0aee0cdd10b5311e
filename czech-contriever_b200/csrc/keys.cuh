// keys.cuh -- 64-bit sortable (score,row) keys shared by every selection kernel.
//
//   key = order(score) << 32 | (0xFFFFFFFF - row)
// so that a larger key is a better hit: higher score first, and among exactly equal fp32
// scores the LOWER row wins -- the survivor rule of faiss's strict `threshold < score`
// insertion test when rows are scanned in ascending order (SURVEY.md 3.2).
// order(NaN) = 0 is reserved: faiss never returns a NaN score, neither do we.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2ip {

__host__ __device__ __forceinline__ uint32_t order_f32(float s) {
    if (s != s) return 0u;
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(s);
#else
    union { float f; uint32_t u; } cv; cv.f = s; uint32_t b = cv.u;
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float unorder_f32(uint32_t o) {
    uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    union { float f; uint32_t u; } cv; cv.u = b; return cv.f;
#endif
}
__host__ __device__ __forceinline__ unsigned long long make_key(float s, uint32_t row) {
    return (static_cast<unsigned long long>(order_f32(s)) << 32) | (0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ uint32_t key_row(unsigned long long k) {
    return 0xFFFFFFFFu - static_cast<uint32_t>(k & 0xFFFFFFFFull);
}
__host__ __device__ __forceinline__ float key_score(unsigned long long k) {
    return unorder_f32(static_cast<uint32_t>(k >> 32));
}

// Allowed-row bitmap of a filtered search (b2ip_search_filtered): bit r & 31 of word r >> 5 is
// set when local row r may be returned.
__device__ __forceinline__ uint32_t row_word(const uint32_t* allow, uint32_t row) {
    return __ldg(allow + (row >> 5));
}
__device__ __forceinline__ bool row_allowed(const uint32_t* allow, long long row) {
    return (__ldg(allow + (row >> 5)) >> (row & 31)) & 1u;
}

}  // namespace b2ip
