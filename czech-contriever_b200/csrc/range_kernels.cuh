// range_kernels.cuh -- range search: every row whose exact score is above a radius r
// (faiss IndexFlatIP::range_search).  DESIGN.md 4.1f.
//
// The coarse kernels run unchanged with the fixed per-query threshold thr = rd(r - eps_q): every
// row with exact score s > r has coarse score c >= s - eps_q > r - eps_q >= thr, so it is admitted.
// After every slab range_drain_kernel rescores the admitted rows exactly, keeps s > r and stores
// them sorted by row; a (query, slab) whose list overflowed goes to range_dense_kernel instead.
// range_gather_kernel finally writes the CSR answer in query order.
//
// Exact scores use the arithmetic of the rescore in finalize_kernel<true, kRows>: lane L handles
// the 16-byte chunks c = L, L + 32, ... of the stored row, each chunk's products summed four at a
// time in fp32 (one multiply, three FMAs), the partials accumulated in fp64 in chunk order, then
// warp_sum(double) and a cast to float.  The same (query, row) therefore gets the same bits from
// the drain, the dense path and b2ip_search.
#pragma once
#include "select_kernels.cuh"

namespace b2ip {

constexpr int RANGE_TILE = 256;            // rows per tile of the dense path (8 warps x 32 rows)
enum { RS_CURSOR = 0,                      // entries of the hit pool in use
       RS_MAX_CNT = 1,                     // largest fill counter of the last slab
       RS_OVERFLOW = 2,                    // lists of the last slab that overflowed
       RS_COUNT = 3 };

// a hit held between slabs: local row on top (so the keys of one query sort by row), score bits below
__device__ __forceinline__ unsigned long long range_hit(float s, uint32_t row) {
    return (static_cast<unsigned long long>(row) << 32) | __float_as_uint(s);
}

__device__ __forceinline__ float range_dot4(float4 a, float4 b) {
    float t = a.x * b.x;
    t = fmaf(a.y, b.y, t);
    t = fmaf(a.z, b.z, t);
    return fmaf(a.w, b.w, t);
}

// This lane's fp64 partial of q . row for NQ queries at once (q4 + b * q_stride4 = query b as float4s,
// in shared memory).  Per query the order of operations is finalize_kernel's.
template <int kRows, int NQ>
__device__ __forceinline__ void range_lane_dots(const uint4* __restrict__ row, const float4* q4, int q_stride4,
                                                int n_chunks, int d, int lane, double (&acc)[NQ]) {
    constexpr int kSh = kRows == ROWS_F16 ? SH_F16 : SH_BF16;
#pragma unroll
    for (int b = 0; b < NQ; b++) acc[b] = 0.0;
#pragma unroll 2
    for (int c = lane; c < n_chunks; c += 32) {
        const uint4 v = row[c];
        if constexpr (kRows == ROWS_F32) {
            const float4 x = make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
#pragma unroll
            for (int b = 0; b < NQ; b++) acc[b] += static_cast<double>(range_dot4(x, q4[b * q_stride4 + c]));
        } else {
            const float2 e0 = unpack2_t<kSh>(v.x), e1 = unpack2_t<kSh>(v.y);
            const float2 e2 = unpack2_t<kSh>(v.z), e3 = unpack2_t<kSh>(v.w);
            const float4 lo = make_float4(e0.x, e0.y, e1.x, e1.y), hi = make_float4(e2.x, e2.y, e3.x, e3.y);
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int b = 0; b < NQ; b++) {
                const float4 qa = (8 * c < d) ? q4[b * q_stride4 + 2 * c] : z;
                const float4 qb = (8 * c + 4 < d) ? q4[b * q_stride4 + 2 * c + 1] : z;
                acc[b] += static_cast<double>(range_dot4(lo, qa));
                acc[b] += static_cast<double>(range_dot4(hi, qb));
            }
        }
    }
}

// thr[q] = rd(radius - eps_q): the admission threshold of the coarse kernels (strict >).  An
// unusable bound (eps_q = inf) gives -inf; range_drain_kernel sends such a query to the dense path.
__global__ void range_threshold_kernel(const float* __restrict__ eps2, float* __restrict__ thr, int nq, float radius) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    float t = __fsub_rd(radius, 0.5f * eps2[q]);
    if (!(t == t)) t = -INFINITY;
    thr[q] = t;
}

struct RangeDrainParams {
    int cap, d, n_chunks;
    long long row_bytes;
    const char* rows;                 // x32 or x16
    const float* q32;                 // [nqb, d] the batch's queries
    const float* eps2;                // [nqb]
    unsigned long long* cand;         // [nqb, cap] the slab's admitted keys (make_key)
    int* cnt;                         // [nqb] fill counters: reset to 0 for the next slab
    int* flags;                       // [nqb] <- FLAG_OVERFLOW: this (query, slab) takes the dense path
    float radius;
    unsigned long long* pool;         // hits of the whole call; room for cap more per query
    long long* tab_off;               // [nqb] this slab's entries: first hit in the pool
    int* tab_cnt;                     //       and number of hits
    long long* rstat;                 // [RS_COUNT]
    long long* gstats;                // GS_CANDIDATES, GS_RESCORED, GS_MAX_ERR, GS_VIOLATIONS
};

// One CTA per query: rescore the query's list of this slab, keep s > radius sorted by row.
// Dynamic shared memory: [cap hit keys | query fp32 [d]].
template <int kRows>
__global__ void __launch_bounds__(SEL_THREADS) range_drain_kernel(const __grid_constant__ RangeDrainParams p) {
    extern __shared__ __align__(16) uint8_t rsm[];
    unsigned long long* hits = reinterpret_cast<unsigned long long*>(rsm);
    float* sq = reinterpret_cast<float*>(rsm + static_cast<size_t>(p.cap) * sizeof(unsigned long long));
    __shared__ int s_m;
    __shared__ long long s_base;
    __shared__ unsigned int s_err, s_viol;
    const int slot = blockIdx.x;
    const int c = p.cnt[slot];
    const float eps2 = p.eps2[slot];
    const bool overflow = c > p.cap || !(eps2 <= FLT_MAX);
    if (threadIdx.x == 0) {
        atomicMax(reinterpret_cast<unsigned long long*>(p.rstat + RS_MAX_CNT), static_cast<unsigned long long>(c));
        atomicAdd(reinterpret_cast<unsigned long long*>(p.gstats + GS_CANDIDATES), static_cast<unsigned long long>(c));
        p.flags[slot] = overflow ? FLAG_OVERFLOW : 0;
        if (overflow) {
            atomicAdd(reinterpret_cast<unsigned long long*>(p.rstat + RS_OVERFLOW), 1ull);
            p.tab_off[slot] = 0;
            p.tab_cnt[slot] = 0;
        }
        s_m = 0; s_err = 0u; s_viol = 0u;
    }
    if (overflow) {
        __syncthreads();                               // (every thread has read cnt)
        if (threadIdx.x == 0) p.cnt[slot] = 0;
        return;
    }
    for (int j = threadIdx.x; j < p.d; j += blockDim.x) sq[j] = p.q32[static_cast<long long>(slot) * p.d + j];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const unsigned long long* keys = p.cand + static_cast<long long>(slot) * p.cap;
    const float cert_eps = 0.5f * eps2;
    const bool cert = cert_eps > 0.f;
    const float inv_cert_eps = cert ? 1.0f / cert_eps : 0.f;
    float w_err = 0.f;
    unsigned int w_viol = 0u;
    for (int i = warp; i < c; i += nw) {
        const unsigned long long key = keys[i];
        const uint32_t row = key_row(key);
        double acc[1];
        range_lane_dots<kRows, 1>(reinterpret_cast<const uint4*>(p.rows + static_cast<long long>(row) * p.row_bytes),
                                  reinterpret_cast<const float4*>(sq), 0, p.n_chunks, p.d, lane, acc);
        const float s = static_cast<float>(warp_sum(acc[0]));
        if (lane == 0) {
            if (cert) {
                const float e = fabsf(key_score(key) - s);
                if (e <= FLT_MAX) {                    // NaN / inf scores carry no margin (see shadow_rows_kernel)
                    const float ratio = e * inv_cert_eps;
                    w_err = fmaxf(w_err, ratio);
                    w_viol += ratio > 1.0f ? 1u : 0u;
                }
            }
            if (s > p.radius) hits[atomicAdd(&s_m, 1)] = range_hit(s, row);
        }
    }
    if (lane == 0) {
        if (w_err > 0.f) atomicMax(&s_err, __float_as_uint(w_err));
        if (w_viol) atomicAdd(&s_viol, w_viol);
    }
    __syncthreads();
    const int m = s_m;
    int P = 2;
    while (P < m) P <<= 1;
    for (int i = m + threadIdx.x; i < P; i += blockDim.x) hits[i] = 0ull;
    if (threadIdx.x == 0) {
        s_base = static_cast<long long>(atomicAdd(reinterpret_cast<unsigned long long*>(p.rstat + RS_CURSOR),
                                                  static_cast<unsigned long long>(m)));
        p.tab_cnt[slot] = m;
        atomicAdd(reinterpret_cast<unsigned long long*>(p.gstats + GS_RESCORED), static_cast<unsigned long long>(c));
        if (s_err) atomicMax(reinterpret_cast<unsigned long long*>(p.gstats + GS_MAX_ERR), static_cast<unsigned long long>(s_err));
        if (s_viol) atomicAdd(reinterpret_cast<unsigned long long*>(p.gstats + GS_VIOLATIONS), static_cast<unsigned long long>(s_viol));
    }
    __syncthreads();
    if (m > 1) block_bitonic_desc(hits, P);            // (rows are distinct: the padding zeros sort last)
    const long long base = s_base;
    for (int j = threadIdx.x; j < m; j += blockDim.x) p.pool[base + m - 1 - j] = hits[j];   // ascending rows
    if (threadIdx.x == 0) {
        p.tab_off[slot] = base;
        p.cnt[slot] = 0;
    }
}

struct RangeDenseParams {
    int d, n_chunks;
    long long row_bytes;
    const char* rows;                 // x32 or x16
    const float* q32;                 // queries, indexed by qlist
    const int* qlist;                 // [nql]
    int nql, n_groups;                // groups of EXACT_QB queries
    long long row0, row1;
    int ntiles;                       // tiles of RANGE_TILE rows in [row0, row1)
    float radius;
    int* counts;                      // [nql, ntiles] hits per (query, tile)          (count pass)
    const long long* offs;            // [nql, ntiles] pool position of the first one   (write pass)
    unsigned long long* pool;
};

// Exact scores of up to EXACT_QB queries against rows [row0, row1), one warp per row, every row read
// once per group.  kWrite = false: count s > radius per (query, tile); true: store those hits at
// offs in ascending row order.  CTA x: query group x % n_groups, tiles x / n_groups, + grid stride
// (CTAs of one wave read the same tiles, from L2).  Dynamic shared memory: EXACT_QB queries [d] fp32.
template <int kRows, bool kWrite>
__global__ void __launch_bounds__(256) range_dense_kernel(const __grid_constant__ RangeDenseParams p) {
    extern __shared__ __align__(16) float dsq[];
    __shared__ int s_cnt[8][EXACT_QB];
    const int g = blockIdx.x % p.n_groups;
    const int nqg = min(EXACT_QB, p.nql - g * EXACT_QB);
    for (int i = threadIdx.x; i < EXACT_QB * p.d; i += blockDim.x) {
        const int b = i / p.d, j = i - b * p.d;
        dsq[i] = b < nqg ? p.q32[static_cast<long long>(p.qlist[g * EXACT_QB + b]) * p.d + j] : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stride = gridDim.x / p.n_groups;
    for (int t = blockIdx.x / p.n_groups; t < p.ntiles; t += stride) {
        const long long r0 = p.row0 + static_cast<long long>(t) * RANGE_TILE + warp * 32;
        float mine[EXACT_QB];
#pragma unroll
        for (int b = 0; b < EXACT_QB; b++) mine[b] = 0.f;
        for (int i = 0; i < 32 && r0 + i < p.row1; i++) {
            double acc[EXACT_QB];
            range_lane_dots<kRows, EXACT_QB>(reinterpret_cast<const uint4*>(p.rows + (r0 + i) * p.row_bytes),
                                             reinterpret_cast<const float4*>(dsq), p.d / 4, p.n_chunks, p.d, lane, acc);
#pragma unroll
            for (int b = 0; b < EXACT_QB; b++) {
                const float s = static_cast<float>(warp_sum(acc[b]));
                if (lane == i) mine[b] = s;
            }
        }
        const bool valid = r0 + lane < p.row1;
        unsigned int bal[EXACT_QB];
#pragma unroll
        for (int b = 0; b < EXACT_QB; b++) {
            bal[b] = __ballot_sync(0xffffffffu, valid && mine[b] > p.radius);
            if (lane == 0) s_cnt[warp][b] = __popc(bal[b]);
        }
        __syncthreads();
        if (!kWrite) {
            if (threadIdx.x < nqg) {
                int sum = 0;
                for (int w = 0; w < 8; w++) sum += s_cnt[w][threadIdx.x];
                p.counts[static_cast<long long>(g * EXACT_QB + threadIdx.x) * p.ntiles + t] = sum;
            }
        } else {
#pragma unroll
            for (int b = 0; b < EXACT_QB; b++) {
                if (b < nqg && ((bal[b] >> lane) & 1u)) {
                    long long pos = p.offs[static_cast<long long>(g * EXACT_QB + b) * p.ntiles + t];
                    for (int w = 0; w < warp; w++) pos += s_cnt[w][b];
                    pos += __popc(bal[b] & ((1u << lane) - 1u));
                    p.pool[pos] = range_hit(mine[b], static_cast<uint32_t>(r0 + lane));
                }
            }
        }
        __syncthreads();
    }
}

// One CTA per listed query: exclusive scan of its per-tile counts into pool positions (the query's
// hits get a contiguous run at the pool cursor), and its table entry.
__global__ void __launch_bounds__(256) range_scan_kernel(const int* __restrict__ counts, long long* __restrict__ offs,
                                                         int ntiles, const int* __restrict__ qlist,
                                                         long long* __restrict__ tab_off, int* __restrict__ tab_cnt,
                                                         long long* __restrict__ rstat) {
    __shared__ long long s_warp[8];
    __shared__ long long s_carry;
    const int i = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int* c = counts + static_cast<long long>(i) * ntiles;
    long long* o = offs + static_cast<long long>(i) * ntiles;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int t0 = 0; t0 < ntiles; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        const long long v = t < ntiles ? c[t] : 0;
        long long incl = v;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, incl, s);
            if (lane >= s) incl += u;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        long long before = s_carry;
        for (int w = 0; w < warp; w++) before += s_warp[w];
        if (t < ntiles) o[t] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const long long total = s_carry;
        s_carry = static_cast<long long>(atomicAdd(reinterpret_cast<unsigned long long*>(rstat + RS_CURSOR),
                                                   static_cast<unsigned long long>(total)));
        tab_off[qlist[i]] = s_carry;
        tab_cnt[qlist[i]] = static_cast<int>(total);
    }
    __syncthreads();
    const long long base = s_carry;
    for (int t = threadIdx.x; t < ntiles; t += blockDim.x) o[t] += base;
}

// One CTA per query: its hits of every slab, in slab order (= ascending rows), to the CSR arrays,
// with local rows mapped to reported ids as finalize_kernel maps them.
// batches[4 b ..]: first query, queries, slabs and first table entry of query batch b (qb queries each);
// the entry of (slab j, query slot i) of a batch is first + j * queries + i.
__global__ void __launch_bounds__(256) range_gather_kernel(const unsigned long long* __restrict__ pool,
                                                           const long long* __restrict__ tab_off,
                                                           const int* __restrict__ tab_cnt,
                                                           const long long* __restrict__ lims,
                                                           const long long* __restrict__ batches, long long qb,
                                                           long long row_offset, int n_seg,
                                                           const long long* __restrict__ seg_local,
                                                           const long long* __restrict__ seg_delta,
                                                           float* __restrict__ out_s, long long* __restrict__ out_r) {
    const long long q = blockIdx.x;
    const long long* bd = batches + 4 * (q / qb);
    const long long slot = q - bd[0], nqb = bd[1], nslabs = bd[2], first = bd[3];
    long long pos = lims[q];
    for (long long j = 0; j < nslabs; j++) {
        const long long e = first + j * nqb + slot;
        const unsigned long long* src = pool + tab_off[e];
        const int c = tab_cnt[e];
        for (int i = threadIdx.x; i < c; i += blockDim.x) {
            const unsigned long long h = src[i];
            long long r = static_cast<long long>(h >> 32);
            if (n_seg > 0) {
                int lo = 0, hi = n_seg - 1;            // last segment starting at or before r
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (seg_local[mid] <= r) lo = mid; else hi = mid - 1;
                }
                r += seg_delta[lo];
            } else {
                r += row_offset;
            }
            out_s[pos + i] = __uint_as_float(static_cast<uint32_t>(h & 0xFFFFFFFFull));
            out_r[pos + i] = r;
        }
        pos += c;
    }
}

}  // namespace b2ip
